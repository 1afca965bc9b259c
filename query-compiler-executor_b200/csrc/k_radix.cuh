// k_radix.cuh -- tuple build, digit histograms and the one-sweep LSD radix pass.
//
// Replaces allocate_relation / allocate_relation_mid_results
// (src/join.c:96-142), build_histogram / build_psum / build_reordered_array
// (src/utilities.c:20-70), iterative_sort (src/join.c:5-94) and the
// quicksort leaves (src/quicksort.c:54-64) of the reference.
//
// The reference sorts 16-byte AoS tuples MSD-first through 8 byte levels
// (4 of them whole-array no-ops when keys < 2^32) and finishes buckets of
// < 4096 tuples with an unstable randomized quicksort.  Here:
//   * a run is packed to one 8-byte word (key << 32 | rowid) whenever the
//     source column's maximum is < 2^32 (known from the load-time column
//     statistics), halving the bytes every pass moves; wider keys use SoA
//     uint64 keys + uint32 ids;
//   * only the ceil(bitlen(max key)/8) significant digits are sorted;
//   * each digit is one kernel that reads every tuple once and writes it once
//     ("one sweep"): per-tile digit counts are published to a status array and
//     the tile's global offsets come from a decoupled look-back over the
//     preceding tiles, so there is no separate per-pass counting kernel;
//   * ranks inside a tile come from warp match/popc (stable), tuples are
//     staged in shared memory in digit order and leave in coalesced runs.
// The sort is stable, so equal keys keep their input order (the reference's
// tie order is unspecified, SURVEY.md 8a-8/9).
//
// Algorithmic HBM bytes: 8 B/tuple once (histogram) + 16 B/tuple/pass packed
// (32 B/tuple/pass for the reference's 16-byte tuples; 24 B wide SoA here).
#pragma once
#include "qce_common.cuh"

#define QCE_RADIX_BITS 8
#define QCE_RADIX_BINS 256  // 8-bit digits: the default
#define QCE_MAX_BINS 512    // 9-bit digits, when they save a pass
#define QCE_MAX_PASSES 8

template <typename KeyT> __device__ __forceinline__ KeyT ld_stream_key(const KeyT *p);
template <> __device__ __forceinline__ u64 ld_stream_key<u64>(const u64 *p) { return ld_stream_u64(p); }
template <> __device__ __forceinline__ u32 ld_stream_key<u32>(const u32 *p) { return ld_stream_u32(p); }

struct RadixShifts {
    int npass;
    int shift[QCE_MAX_PASSES];
};

// ---- tuple build ---------------------------------------------------------------
// Packed, from a base column: out[i] = col[i] << 32 | i   (src/join.c:131-134)
// HIST: also count the top 8 key bits (key >> hist_shift) into ghist[256] -- level A of the
// MSD sort and the exchange's splitter histogram, taken while the keys stream through
// anyway instead of in a pass of its own (8 B/tuple saved).
template <bool HIST>
__global__ void __launch_bounds__(256)
k_build_packed_base(const u64 *__restrict__ col, u64 n, u64 *__restrict__ out, u64 id_base, int hist_shift,
                    u32 *__restrict__ ghist)
{
    // id_base: first row id of the window when a rank builds only its row range
    __shared__ u32 sh[HIST ? 256 : 1];
    if (HIST) { sh[threadIdx.x] = 0; __syncthreads(); }
    const u64 stride = (u64)gridDim.x * 512;
    for (u64 e = ((u64)blockIdx.x * 256 + threadIdx.x) * 2; e < n; e += stride) {
        if (e + 1 < n) {
            u64 a, b;
            ld_stream_u64x2(col + e, a, b);
            st_stream_u64x2(out + e, (a << 32) | (e + id_base), (b << 32) | (e + 1 + id_base));
            if (HIST) { atomicAdd(&sh[(u32)(a >> hist_shift) & 255u], 1u); atomicAdd(&sh[(u32)(b >> hist_shift) & 255u], 1u); }
        } else {
            const u64 a = col[e];
            out[e] = (a << 32) | (e + id_base);
            if (HIST) atomicAdd(&sh[(u32)(a >> hist_shift) & 255u], 1u);
        }
    }
    if (HIST) {
        __syncthreads();
        if (sh[threadIdx.x]) atomicAdd(&ghist[threadIdx.x], sh[threadIdx.x]);
    }
}
// Packed, through a row-id column: out[i] = col[ids[i]] << 32 | ids[i]
// (src/join.c:107-112).  The gather is sector-bound unless ids are clustered
// (filter outputs are ascending).
// POS: the payload is the element's POSITION in the row-id column instead of the row id, so
// that the columns aligned with it can be gathered after the merge (SURVEY.md 8f-2).
template <bool HIST, bool POS = false>
__global__ void __launch_bounds__(256)
k_build_packed_ids(const __grid_constant__ ColRef col, const u32 *__restrict__ ids, u64 n,
                   u64 *__restrict__ out, int hist_shift, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[HIST ? 256 : 1];
    if (HIST) { sh[threadIdx.x] = 0; __syncthreads(); }
    const u64 stride = (u64)gridDim.x * 256 * 4;
    for (u64 i0 = (u64)blockIdx.x * 256 * 4 + threadIdx.x; i0 < n; i0 += stride) {
        u32 id[4];
        u64 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) id[k] = (i0 + k * 256 < n) ? ids[i0 + k * 256] : 0;
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = (i0 + k * 256 < n) ? col(id[k]) : 0;
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (i0 + k * 256 < n) {
                out[i0 + k * 256] = (v[k] << 32) | (POS ? (u64)(i0 + k * 256) : (u64)id[k]);
                if (HIST) atomicAdd(&sh[(u32)(v[k] >> hist_shift) & 255u], 1u);
            }
    }
    if (HIST) {
        __syncthreads();
        if (sh[threadIdx.x]) atomicAdd(&ghist[threadIdx.x], sh[threadIdx.x]);
    }
}
// Wide (keys may exceed 32 bits): SoA keys[] / ids[].
__global__ void __launch_bounds__(256)
k_build_wide(const __grid_constant__ ColRef col, const u32 *__restrict__ ids, u64 n,
             u64 *__restrict__ keys, u32 *__restrict__ out_ids, u32 id_base)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        u32 id = ids ? ids[i] : (u32)i + id_base;
        keys[i] = col(id);
        out_ids[i] = id;
    }
}
// Packed from two row-id columns: out[i] = hi[i] << 32 | (lo ? lo[i] : 0).
// Used by the bystander re-join (R' = (key=last[i], payload=edit[i]),
// S' = (key=driver[i], 0); src/join.c:431-442) and the distinct-pair pass.
__global__ void __launch_bounds__(256)
k_pack_pairs(const u32 *__restrict__ hi, const u32 *__restrict__ lo, u64 n, u64 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride)
        out[i] = ((u64)hi[i] << 32) | (lo ? (u64)lo[i] : 0ull);
}
__global__ void __launch_bounds__(256)
k_unpack_lo(const u64 *__restrict__ in, u64 n, u32 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) out[i] = (u32)in[i];
}

// ---- digit histograms of every pass in one read (build_histogram,
// src/utilities.c:20-31, hoisted out of the per-bucket loop) ------------------------
// `bins` = 256 or 512 (8- or 9-bit digits), the same for every pass of a sort.
__global__ void __launch_bounds__(512)
k_radix_hist(const u64 *__restrict__ keys, u64 n, RadixShifts rs, u32 bins, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[QCE_MAX_PASSES * QCE_MAX_BINS];
    const u32 mask = bins - 1;
    for (u32 i = threadIdx.x; i < rs.npass * bins; i += 512) sh[i] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * 1024;
    for (u64 e = ((u64)blockIdx.x * 512 + threadIdx.x) * 2; e < n; e += stride) {
        u64 a, b = 0;
        const bool two = e + 1 < n;
        if (two) ld_stream_u64x2(keys + e, a, b);
        else a = keys[e];
#pragma unroll
        for (int p = 0; p < QCE_MAX_PASSES; p++) {
            if (p < rs.npass) {
                atomicAdd(&sh[p * bins + ((u32)(a >> rs.shift[p]) & mask)], 1u);
                if (two) atomicAdd(&sh[p * bins + ((u32)(b >> rs.shift[p]) & mask)], 1u);
            }
        }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < rs.npass * bins; i += 512)
        if (sh[i]) atomicAdd(&ghist[i], sh[i]);
}

// One-digit histogram of 32-bit keys (row ids), for the bucketed checksum.
__global__ void __launch_bounds__(512)
k_hist_u32(const u32 *__restrict__ keys, u64 n, u32 base, int shift, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[256];
    if (threadIdx.x < 256) sh[threadIdx.x] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * 2048;
    const u64 n4 = n & ~3ull;
    for (u64 e = ((u64)blockIdx.x * 512 + threadIdx.x) * 4; e < n4; e += stride) {
        uint4 k = ld_stream_u32x4(keys + e);
        atomicAdd(&sh[((k.x - base) >> shift) & 255], 1u);
        atomicAdd(&sh[((k.y - base) >> shift) & 255], 1u);
        atomicAdd(&sh[((k.z - base) >> shift) & 255], 1u);
        atomicAdd(&sh[((k.w - base) >> shift) & 255], 1u);
    }
    if (blockIdx.x == 0 && threadIdx.x < (n - n4)) atomicAdd(&sh[((keys[n4 + threadIdx.x] - base) >> shift) & 255], 1u);
    __syncthreads();
    if (threadIdx.x < 256 && sh[threadIdx.x]) atomicAdd(&ghist[threadIdx.x], sh[threadIdx.x]);
}

// build_psum (src/utilities.c:34-48): exclusive prefix over the bins of each
// pass.  One CTA of `bins` (256 or 512) threads per pass.
__global__ void __launch_bounds__(512) k_radix_bases(const u32 *__restrict__ ghist, u32 *__restrict__ gbase)
{
    __shared__ u32 scratch[33];
    const u32 bins = blockDim.x;
    u32 v = ghist[blockIdx.x * bins + threadIdx.x];
    // block_scan_excl is written for a compile-time thread count; 16 warps cover both sizes
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 incl = warp_scan_incl<u32>(v);
    if (lane == 31) scratch[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        u32 w = (lane < (int)(bins / 32)) ? scratch[lane] : 0u;
        u32 wi = warp_scan_incl<u32>(w);
        scratch[lane] = wi - w;
    }
    __syncthreads();
    gbase[blockIdx.x * bins + threadIdx.x] = scratch[warp] + incl - v;
}

// ---- digit functors ------------------------------------------------------------
// A functor returns the digit of a key under a `mask` (bins - 1) the kernel supplies.
struct DigitShift {
    int shift;
    __device__ __forceinline__ u32 operator()(u64 k, u32 mask) const { return (u32)(k >> shift) & mask; }
    __device__ __forceinline__ u32 operator()(u32 k, u32 mask) const { return (k >> shift) & mask; }
};
// Packed words always sort key bits, i.e. word bits >= 32: the digit only needs
// the high register (no 64-bit funnel shifts).  hi_shift = shift - 32.
struct DigitShiftHi {
    int hi_shift;
    __device__ __forceinline__ u32 operator()(u64 k, u32 mask) const { return ((u32)(k >> 32) >> hi_shift) & mask; }
};
// Range partition for the multi-GPU exchange.  Splitters sit on the boundaries of
// the 256-bin histogram of the top 8 significant key bits, so the destination of
// a tuple is a table lookup on those bits (4 destinations per table word).
struct DigitSplit {
    const u32 *lut; // device memory, 256 x uint8: histogram bin -> destination rank.  Not a
                    // kernel-parameter array: lanes index it divergently, which the
                    // constant bank serialises; 256 B in global memory stay in L1.
    int shift;      // 32 + key_bits - 8 (packed word)
    __device__ __forceinline__ u32 operator()(u64 k, u32) const
    {
        const u32 bin = (u32)(k >> shift) & 255u;
        return (__ldg(lut + (bin >> 2)) >> ((bin & 3u) * 8)) & 255u;
    }
};

// Lanes of the warp holding the same BITS-bit digit.  `match.any` gives this in
// one instruction, but on sm_100a it runs on the address-divergence unit at about
// one warp instruction per 60 cycles per SM (ncu: pipe_adu 73 % busy, the pass
// capped at ~2 TB/s).  One ballot per digit bit, intersected, goes through the
// vote path at two warps per clock instead.
template <int BITS> __device__ __forceinline__ u32 warp_peers(u32 d)
{
    // per bit: test -> predicate, ballot m, then keep the lanes whose bit agrees
    // with ours: peers &= m ^ (bit ? 0 : ~0).  Hand-written: the compiler's
    // version of the plain C loop cost ~7 instructions per bit; this is 2-3.
    u32 peers = QCE_FULL_MASK;
#pragma unroll
    for (int b = 0; b < BITS; b++) {
        asm("{\n\t"
            ".reg .pred p;\n\t"
            ".reg .b32 t, m, nm;\n\t"
            "and.b32 t, %1, %2;\n\t"
            "setp.ne.u32 p, t, 0;\n\t"
            "vote.sync.ballot.b32 m, p, 0xffffffff;\n\t"
            "selp.b32 nm, 0, 0xffffffff, p;\n\t"
            "lop3.b32 %0, %0, m, nm, 0x60;\n\t" // a & (b ^ c)
            "}"
            : "+r"(peers)
            : "r"(d), "r"(1u << b));
    }
    return peers;
}

// ---- one-sweep pass ------------------------------------------------------------
// Tile status word: top 2 bits = flag, low 30 bits = count (n < 2^30 per sort).
#define QCE_ST_PART 0x40000000u
#define QCE_ST_INCL 0x80000000u
#define QCE_ST_MASK 0x3fffffffu

template <int THREADS, int ITEMS, int BITS, typename KeyT = u64> struct OnesweepSmem {
    static constexpr int BINS = 1 << BITS;
    u32 warp_hist[(THREADS / 32) * BINS]; // per-warp digit counts -> bases
    u32 tile_excl[BINS];                  // digit start inside the sorted tile
    u32 goff[BINS];                       // global start of digit minus tile_excl
    u32 scratch[33];
    u32 tile_id;
    KeyT keys[THREADS * ITEMS];
};

// One tile of the pass.  FULL = every slot of the tile holds a real tuple (no
// bounds checks, no padding logic): all tiles but the last.
template <int THREADS, int ITEMS, int BITS, bool HAS_VALS, bool FULL, int MATCH_EVERY, typename KeyT,
          typename DigitOp>
__device__ __forceinline__ void
onesweep_tile(OnesweepSmem<THREADS, ITEMS, BITS, KeyT> &sm, u32 *svals, const KeyT *__restrict__ keys_in,
              KeyT *__restrict__ keys_out, const u32 *__restrict__ vals_in, u32 *__restrict__ vals_out, u32 n,
              const DigitOp &digit, const u32 *__restrict__ gbase, u32 *__restrict__ status, u32 tile)
{
    constexpr int TILE = THREADS * ITEMS;
    constexpr int WARPS = THREADS / 32;
    constexpr int BINS = 1 << BITS;
    constexpr u32 DMASK = BINS - 1;
    constexpr int BPT = (BINS + THREADS - 1) / THREADS; // bins per thread, consecutive
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 tbase = tile * TILE;
    const u32 nvalid = FULL ? (u32)TILE : (n - tbase);
    const u32 npad = TILE - nvalid; // padding slots of the last tile (digit BINS-1)

    // ---- load: warp-striped so that (warp, item, lane) order == input order
    KeyT key[ITEMS];
    u32 val[HAS_VALS ? ITEMS : 1];
    const u32 wbase = tbase + warp * (32 * ITEMS) + lane;
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 idx = wbase + j * 32;
        if (FULL || idx < n) {
            key[j] = ld_stream_key<KeyT>(keys_in + idx);
            if (HAS_VALS) val[j] = ld_stream_u32(vals_in + idx);
        } else {
            key[j] = (KeyT)~(KeyT)0;
            if (HAS_VALS) val[j] = 0u;
        }
    }

    // ---- rank inside the warp.  Lanes with the same digit are found with
    // per-bit ballots (warp_peers); the lowest of them reserves the group's slots
    // with one shared atomicAdd (program order within the warp keeps items in
    // input order) and hands the base to its peers.  Done in chunks of CH items
    // with the three long-latency steps (ballots, ATOMS, SHFL) each issued back
    // to back, so their latencies overlap instead of adding up.
    u32 rd[ITEMS]; // digit << 16 | rank inside (warp, digit)
    u32 *wh = sm.warp_hist + warp * BINS;
    const u32 lt = lanemask_lt();
    constexpr int CH = (ITEMS % 4 == 0) ? 4 : ((ITEMS % 3 == 0) ? 3 : 1);
#pragma unroll
    for (int j0 = 0; j0 < ITEMS; j0 += CH) {
        u32 d[CH], peers[CH], old[CH];
#pragma unroll
        for (int c = 0; c < CH; c++) {
            // padding of the last tile must sort behind every real tuple of the tile
            d[c] = (!FULL && (wbase + (j0 + c) * 32) >= n) ? DMASK : digit(key[j0 + c], DMASK);
            // every MATCH_EVERY-th item goes to match.any: the ADU pipe is idle
            // otherwise, so it takes a share of the ranking off the ALU ballots
            peers[c] = (MATCH_EVERY > 0 && ((j0 + c) % (MATCH_EVERY > 0 ? MATCH_EVERY : 1)) == MATCH_EVERY - 1)
                           ? __match_any_sync(QCE_FULL_MASK, d[c])
                           : warp_peers<BITS>(d[c]);
        }
#pragma unroll
        for (int c = 0; c < CH; c++) {
            old[c] = 0;
            if ((peers[c] & lt) == 0) old[c] = atomicAdd(&wh[d[c]], (u32)__popc(peers[c]));
        }
#pragma unroll
        for (int c = 0; c < CH; c++) {
            old[c] = __shfl_sync(QCE_FULL_MASK, old[c], __ffs(peers[c]) - 1);
            rd[j0 + c] = (d[c] << 16) | (old[c] + __popc(peers[c] & lt));
        }
    }
    __syncthreads(); // all warps have ranked

    // ---- per digit (thread t owns bins t*BPT .. t*BPT+BPT-1): exclusive scan of
    //      the warp counts, tile total, publish the tile-local count
    u32 cnt[BPT], sum = 0;
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        const int b = tid * BPT + q;
        cnt[q] = 0;
        if (b < BINS) {
            u32 run = 0;
#pragma unroll
            for (int w = 0; w < WARPS; w++) {
                const u32 c = sm.warp_hist[w * BINS + b];
                sm.warp_hist[w * BINS + b] = run;
                run += c;
            }
            cnt[q] = run;
            // the padding of the last tile is not part of the global count
            const u32 pub = run - ((!FULL && b == BINS - 1) ? npad : 0u);
            st_relaxed_gpu_u32(status + (size_t)tile * BINS + b, (tile == 0 ? QCE_ST_INCL : QCE_ST_PART) | pub);
        }
        sum += cnt[q];
    }
    // ---- digit starts inside the tile (exclusive scan over the bins)
    {
        u32 tot;
        u32 ex = block_scan_excl<u32, THREADS>(sum, sm.scratch, &tot);
#pragma unroll
        for (int q = 0; q < BPT; q++) {
            const int b = tid * BPT + q;
            if (b < BINS) sm.tile_excl[b] = ex;
            ex += cnt[q];
        }
    }
    // ---- decoupled look-back: sum the counts of the preceding tiles.  The status
    //      words of LB predecessors are fetched together (one L2 round trip).
#pragma unroll
    for (int q = 0; q < BPT; q++) {
        const int b = tid * BPT + q;
        if (b < BINS) {
            u32 excl = 0;
            if (tile > 0) {
                const u32 pub = cnt[q] - ((!FULL && b == BINS - 1) ? npad : 0u);
                constexpr int LB = 4;
                int p = (int)tile - 1;
                bool done = false;
                while (!done) {
                    u32 v[LB];
#pragma unroll
                    for (int k = 0; k < LB; k++)
                        v[k] = (p - k >= 0) ? ld_relaxed_gpu_u32(status + (size_t)(p - k) * BINS + b)
                                            : QCE_ST_INCL; // before tile 0: inclusive prefix 0
                    int used = 0;
#pragma unroll
                    for (int k = 0; k < LB; k++) {
                        if (!done && used == k && (v[k] & ~QCE_ST_MASK) != 0) {
                            excl += v[k] & QCE_ST_MASK;
                            done = (v[k] & QCE_ST_INCL) != 0;
                            used = k + 1;
                        }
                    }
                    p -= used; // resume at the first tile that had not published yet
                    if (!done && used < LB) __nanosleep(20);
                }
                st_relaxed_gpu_u32(status + (size_t)tile * BINS + b, QCE_ST_INCL | (excl + pub));
            }
            sm.goff[b] = gbase[b] + excl - sm.tile_excl[b];
        }
    }
    __syncthreads();

    // ---- stage in shared memory in digit order
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 d = rd[j] >> 16;
        const u32 pos = sm.tile_excl[d] + wh[d] + (rd[j] & 0xffffu);
        sm.keys[pos] = key[j];
        if (HAS_VALS) svals[pos] = val[j];
    }
    __syncthreads();

    // ---- coalesced write-out: consecutive threads, consecutive slots of a digit
    //      (positions >= nvalid are exactly the padding of the last tile)
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 p = tid + j * THREADS;
        if (FULL || p < nvalid) {
            const KeyT k = sm.keys[p];
            const u32 g = sm.goff[digit(k, DMASK)] + p;
            keys_out[g] = k;
            if (HAS_VALS) vals_out[g] = svals[p];
        }
    }
}

template <int THREADS, int ITEMS, int MIN_CTAS, int BITS, int MATCH_EVERY, bool HAS_VALS, typename KeyT,
          typename DigitOp>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
k_onesweep(const KeyT *__restrict__ keys_in, KeyT *__restrict__ keys_out,
           const u32 *__restrict__ vals_in, u32 *__restrict__ vals_out, u32 n, DigitOp digit,
           const u32 *__restrict__ gbase, u32 *__restrict__ status, u32 *__restrict__ tile_counter)
{
    static_assert(THREADS * ITEMS <= 65536 && ITEMS * 32 < 65536, "tile shape");
    constexpr int TILE = THREADS * ITEMS;
    constexpr int WARPS = THREADS / 32;
    constexpr int BINS = 1 << BITS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef OnesweepSmem<THREADS, ITEMS, BITS, KeyT> Smem;
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
    u32 *svals = reinterpret_cast<u32 *>(smem_raw + sizeof(Smem));

    // Tiles are claimed in launch order so that every tile a CTA may wait on in
    // the look-back is owned by a CTA that is already resident.
    if (threadIdx.x == 0) sm.tile_id = atomicAdd(tile_counter, 1u);
    for (int i = threadIdx.x; i < WARPS * BINS; i += THREADS) sm.warp_hist[i] = 0;
    __syncthreads();
    const u32 tile = sm.tile_id;
    if ((tile + 1) * (u32)TILE <= n)
        onesweep_tile<THREADS, ITEMS, BITS, HAS_VALS, true, MATCH_EVERY, KeyT>(sm, svals, keys_in, keys_out, vals_in,
                                                                              vals_out, n, digit, gbase, status, tile);
    else
        onesweep_tile<THREADS, ITEMS, BITS, HAS_VALS, false, MATCH_EVERY, KeyT>(sm, svals, keys_in, keys_out, vals_in,
                                                                               vals_out, n, digit, gbase, status, tile);
}

// ---- small runs: whole sort in one CTA's shared memory --------------------------
// Replaces the reference's small-bucket sort (random_quicksort, src/quicksort.c:
// 54-64, used below 4096 tuples -- src/join.c:6,56).  A run of up to THREADS*ITEMS
// tuples is loaded once, every digit pass ranks it with the same ballot scheme as
// k_onesweep and permutes it between two shared-memory buffers, and it is written
// back once: one launch instead of histogram + prefix + one launch per digit (and
// their look-back arrays), which is what bounds the many-small-queries regime.
// Stable, like the large path.
template <int THREADS, int ITEMS, bool HAS_VALS>
__global__ void __launch_bounds__(THREADS)
k_block_sort(u64 *__restrict__ keys, u32 *__restrict__ vals, u32 n, RadixShifts rs)
{
    constexpr int TILE = THREADS * ITEMS;
    constexpr int WARPS = THREADS / 32;
    constexpr int BINS = 256;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64 *skeys = reinterpret_cast<u64 *>(smem_raw);                       // TILE
    u32 *svals = reinterpret_cast<u32 *>(skeys + TILE);                   // TILE (HAS_VALS)
    u32 *warp_hist = svals + (HAS_VALS ? TILE : 0);                       // WARPS * BINS
    u32 *tile_excl = warp_hist + WARPS * BINS;                            // BINS
    u32 *scratch = tile_excl + BINS;                                      // 33
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 lt = lanemask_lt();
    const u32 slot0 = warp * (32 * ITEMS) + lane; // warp-striped: (warp, item, lane) == run order

    u64 key[ITEMS];
    u32 val[HAS_VALS ? ITEMS : 1];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 idx = slot0 + j * 32;
        key[j] = (idx < n) ? keys[idx] : ~0ull; // padding: digit 255 in every pass, stays last
        if (HAS_VALS) val[j] = (idx < n) ? vals[idx] : 0u;
    }
    for (int p = 0; p < rs.npass; p++) {
        const int shift = rs.shift[p];
        for (int i = tid; i < WARPS * BINS; i += THREADS) warp_hist[i] = 0;
        __syncthreads();
        u32 rd[ITEMS];
        u32 *wh = warp_hist + warp * BINS;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 d = (u32)(key[j] >> shift) & 255u;
            const u32 peers = warp_peers<8>(d);
            u32 old = 0;
            if ((peers & lt) == 0) old = atomicAdd(&wh[d], (u32)__popc(peers));
            old = __shfl_sync(QCE_FULL_MASK, old, __ffs(peers) - 1);
            rd[j] = (d << 16) | (old + __popc(peers & lt));
        }
        __syncthreads();
        u32 cnt = 0;
        if (tid < BINS) {
#pragma unroll
            for (int w = 0; w < WARPS; w++) {
                const u32 c = warp_hist[w * BINS + tid];
                warp_hist[w * BINS + tid] = cnt;
                cnt += c;
            }
        }
        u32 tot;
        const u32 ex = block_scan_excl<u32, THREADS>(cnt, scratch, &tot);
        if (tid < BINS) tile_excl[tid] = ex;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 d = rd[j] >> 16;
            const u32 pos = tile_excl[d] + wh[d] + (rd[j] & 0xffffu);
            skeys[pos] = key[j];
            if (HAS_VALS) svals[pos] = val[j];
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            key[j] = skeys[slot0 + j * 32];
            if (HAS_VALS) val[j] = svals[slot0 + j * 32];
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 idx = slot0 + j * 32;
        if (idx < n) {
            keys[idx] = key[j];
            if (HAS_VALS) vals[idx] = val[j];
        }
    }
}

// ---- MSD partition + in-shared-memory bucket sort (large, non-skewed runs) -------
// The reference sorts MSD-first: byte 1, then byte 2 ... per bucket, and hands
// buckets below 4096 tuples to a small sort (iterative_sort, src/join.c:5-94).
// The same shape is the cheapest one here, because an MSD partition does not
// have to be stable: no per-bit ballots, no look-back chain.
//   pass A   scatter by the top P1 key bits          (k_msd_partition, level 0)
//   pass B   per bucket, scatter by the next P2 bits (k_msd_partition, level 1)
//   finish   every sub-bucket (<= 4096 tuples) is sorted on the remaining key
//            bits inside one CTA's shared memory     (k_msd_local_sort)
// Inside a tile a key's slot among equal digits comes from a shared-memory
// cursor (atomicAdd with return); a tile reserves its output range per digit
// with one global atomicAdd on the bucket's cursor.  Equal keys end up in an
// unspecified order (as in the reference, whose quicksort is rand()-driven).
// Skew: if any sub-bucket exceeds the finish kernel's capacity the caller falls
// back to the LSD one-sweep passes, which do not care about key distribution.
#define QCE_MSD_THREADS 256
#define QCE_MSD_ITEMS 16
#define QCE_MSD_TILE (QCE_MSD_THREADS * QCE_MSD_ITEMS)

// tile_start[b] = first tile of bucket b when every bucket is cut into tiles of
// QCE_MSD_TILE (one CTA, nbuckets <= 256 threads); tile_start[nbuckets] = total.
__global__ void __launch_bounds__(256)
k_msd_tile_starts(const u32 *__restrict__ bucket_size, u32 nbuckets, u32 *__restrict__ tile_start)
{
    __shared__ u32 scratch[33];
    const u32 v = threadIdx.x < nbuckets ? (bucket_size[threadIdx.x] + QCE_MSD_TILE - 1) / QCE_MSD_TILE : 0u;
    u32 tot;
    const u32 ex = block_scan_excl<u32, 256>(v, scratch, &tot);
    if (threadIdx.x < nbuckets) tile_start[threadIdx.x] = ex;
    if (threadIdx.x == 0) tile_start[nbuckets] = tot;
}

// Bucket and range of tile `t` (tiles never straddle buckets).
__device__ __forceinline__ bool msd_locate_tile(u32 t, const u32 *__restrict__ tile_start, const u32 *__restrict__ bucket_off,
                                                const u32 *__restrict__ bucket_size, u32 nbuckets, u32 &bucket,
                                                u32 &begin, u32 &count)
{
    if (t >= tile_start[nbuckets]) return false;
    u32 lo = 0, hi = nbuckets; // largest b with tile_start[b] <= t
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (tile_start[mid] <= t) lo = mid; else hi = mid;
    }
    // buckets without tiles share their start with the next one: move to the owner
    while (lo + 1 < nbuckets && tile_start[lo + 1] <= t) lo++;
    bucket = lo;
    const u32 local = (t - tile_start[lo]) * QCE_MSD_TILE;
    begin = bucket_off[lo] + local;
    count = min((u32)QCE_MSD_TILE, bucket_size[lo] - local);
    return true;
}

// Histogram of the level's digit, per bucket: ghist[bucket * bins + digit].
__global__ void __launch_bounds__(QCE_MSD_THREADS)
k_msd_hist(const u64 *__restrict__ keys, const u32 *__restrict__ tile_start, const u32 *__restrict__ bucket_off,
           const u32 *__restrict__ bucket_size, u32 nbuckets, u64 base, int shift, u32 bins, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[256];
    __shared__ u32 s_loc[3];
    if (threadIdx.x == 0) {
        u32 b = 0, beg = 0, cnt = 0;
        if (!msd_locate_tile(blockIdx.x, tile_start, bucket_off, bucket_size, nbuckets, b, beg, cnt)) cnt = 0;
        s_loc[0] = b; s_loc[1] = beg; s_loc[2] = cnt;
    }
    sh[threadIdx.x] = 0;
    __syncthreads();
    const u32 bucket = s_loc[0], begin = s_loc[1], count = s_loc[2];
    if (count == 0) return;
    const u32 mask = bins - 1;
#pragma unroll 4
    for (u32 i = threadIdx.x; i < count; i += QCE_MSD_THREADS)
        atomicAdd(&sh[(u32)((ld_stream_u64(keys + begin + i) - base) >> shift) & mask], 1u);
    __syncthreads();
    if (threadIdx.x < bins && sh[threadIdx.x]) atomicAdd(&ghist[bucket * bins + threadIdx.x], sh[threadIdx.x]);
}

// Rank of a key among the tile's keys with the same digit.  Plain: one shared-memory atomic per key.
// Skewed tiles (a heavy key, or row ids of a heavy key's matches) put most lanes of a warp on one
// counter, which the hardware serialises lane by lane; `agg` (decided per warp from the tile's first
// keys) lets the lanes that share the leader's digit count once and take consecutive slots.
__device__ __forceinline__ u32 msd_rank(u32 *cnt, u32 dg, bool live, bool agg)
{
    if (!agg) return live ? atomicAdd(&cnt[dg], 1u) : 0u;
    const u32 lead = __shfl_sync(QCE_FULL_MASK, live ? dg : 0xffffffffu, 0);
    const u32 same = __ballot_sync(QCE_FULL_MASK, live && dg == lead);
    u32 b = 0;
    if ((threadIdx.x & 31) == 0 && same) b = atomicAdd(&cnt[lead], (u32)__popc(same));
    b = __shfl_sync(QCE_FULL_MASK, b, 0);
    if (live && dg == lead) return b + __popc(same & lanemask_lt());
    return live ? atomicAdd(&cnt[dg], 1u) : 0u;
}
// true when at least a quarter of the warp's lanes share lane 0's digit
__device__ __forceinline__ bool msd_warp_skewed(u32 dg, bool live)
{
    const u32 lead = __shfl_sync(QCE_FULL_MASK, live ? dg : 0xffffffffu, 0);
    return __popc(__ballot_sync(QCE_FULL_MASK, live && dg == lead)) >= 8;
}

// One unstable partition pass.  cursor[bucket * bins + digit] starts at the
// global output offset of that (bucket, digit) range and is advanced by the tiles.
// MIN_CTAS = 4 caps the kernel at 32 registers (100 % occupancy with 512 threads); VEC loads
// two adjacent tuples with one 128-bit load where the tile starts on a 16-byte boundary.
template <int THREADS, int ITEMS, typename KeyT = u64, int MIN_CTAS = (THREADS == 512 ? 3 : 1), bool VEC = false>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
k_msd_partition(const KeyT *__restrict__ in, KeyT *__restrict__ out, const u32 *__restrict__ tile_start,
                const u32 *__restrict__ bucket_off, const u32 *__restrict__ bucket_size, u32 nbuckets, KeyT base,
                int shift, u32 bins, u32 *__restrict__ cursor, const u32 *__restrict__ lut)
{
    static_assert(THREADS * ITEMS == QCE_MSD_TILE && THREADS >= 256, "tile shape");
    __shared__ KeyT skeys[QCE_MSD_TILE];
    __shared__ u32 cnt[256], excl[256], goff[256];
    __shared__ u32 scratch[33];
    __shared__ u32 s_loc[3];
    const int tid = threadIdx.x;
    if (tid == 0) {
        u32 b = 0, beg = 0, c = 0;
        if (!msd_locate_tile(blockIdx.x, tile_start, bucket_off, bucket_size, nbuckets, b, beg, c)) c = 0;
        s_loc[0] = b; s_loc[1] = beg; s_loc[2] = c;
    }
    if (tid < 256) cnt[tid] = 0;
    __syncthreads();
    const u32 bucket = s_loc[0], begin = s_loc[1], count = s_loc[2];
    if (count == 0) return;
    const u32 mask = lut ? 255u : bins - 1;

    KeyT key[ITEMS];
    u32 slot[ITEMS]; // digit << 16 | slot among the tile's keys with that digit
    // element index of item j: strided by THREADS, or (VEC) adjacent pairs strided by 2 * THREADS
    const bool vec = VEC && sizeof(KeyT) == 8 && ((begin & 1u) == 0);
#define MSD_ITEM_INDEX(j) (vec ? (u32)(2 * tid + ((j) & 1) + ((j) >> 1) * 2 * THREADS) : (u32)(tid + (j) * THREADS))
    if (vec) {
#pragma unroll
        for (int j = 0; j < ITEMS; j += 2) {
            const u32 i = MSD_ITEM_INDEX(j);
            if (i + 1 < count) {
                u64 a, b;
                ld_stream_u64x2(reinterpret_cast<const u64 *>(in) + begin + i, a, b);
                key[j] = (KeyT)a;
                key[j + 1] = (KeyT)b;
            } else if (i < count) {
                key[j] = ld_stream_key<KeyT>(in + begin + i);
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 i = tid + j * THREADS;
            if (i < count) key[j] = ld_stream_key<KeyT>(in + begin + i);
        }
    }
    bool agg = false;
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = MSD_ITEM_INDEX(j);
        const bool live = i < count;
        u32 d = 0;
        if (live) {
            d = (u32)((key[j] - base) >> shift) & mask;
            // exchange partition: the digit is a histogram bin, its destination rank comes from a table
            if (lut) d = (__ldg(lut + (d >> 2)) >> ((d & 3u) * 8)) & 255u;
        }
        if (j == 0) agg = bins > 4 && msd_warp_skewed(d, live);
        const u32 r = msd_rank(cnt, d, live, agg);
        if (live) slot[j] = (d << 16) | r;
    }
    __syncthreads();
    {
        const u32 c = tid < 256 ? cnt[tid] : 0u;
        u32 tot;
        const u32 ex = block_scan_excl<u32, THREADS>(c, scratch, &tot);
        if (tid < 256) {
            excl[tid] = ex;
            // reserve this tile's output range of the (bucket, digit) run
            goff[tid] = (c ? atomicAdd(&cursor[bucket * bins + tid], c) : 0u) - ex;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = MSD_ITEM_INDEX(j);
        if (i < count) skeys[excl[slot[j] >> 16] + (slot[j] & 0xffffu)] = key[j];
    }
#undef MSD_ITEM_INDEX
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 p = tid + j * THREADS;
        if (p < count) {
            const KeyT k = skeys[p];
            u32 d = (u32)((k - base) >> shift) & mask;
            if (lut) d = (__ldg(lut + (d >> 2)) >> ((d & 3u) * 8)) & 255u;
            out[goff[d] + p] = k;
        }
    }
}

// ---- the same pass, Blackwell-native data movement --------------------------------------
// Persistent CTAs; the tiles stream into shared memory through the bulk-copy engine
// (cp.async.bulk, 1-D TMA: SASS UBLKCP) and complete on an mbarrier (SYNCS), two tiles in
// flight per CTA: while tile k is ranked, staged and written, tile k+1 is already landing.
// The landing buffer doubles as the staging buffer (once a tile's keys are in registers its
// buffer is free), so a CTA needs 2 x 32 KB and three of them share an SM.  The plain kernel
// above issues its loads at tile start and hides their latency only by CTA co-residency: its
// four phases serialise behind the load (DESIGN.md: issue 51 %, DRAM 51 %, barrier +
// short-scoreboard stalls).
struct MsdTileDesc { u32 bucket, begin, count, pad; };
__global__ void __launch_bounds__(256)
k_msd_tile_desc(const u32 *__restrict__ tile_start, const u32 *__restrict__ bucket_off, const u32 *__restrict__ bucket_size,
                u32 nbuckets, u32 ntiles_cap, MsdTileDesc *__restrict__ desc)
{
    const u32 t = blockIdx.x * 256 + threadIdx.x;
    if (t >= ntiles_cap) return;
    MsdTileDesc d{0u, 0u, 0u, 0u};
    u32 b = 0, beg = 0, c = 0;
    if (msd_locate_tile(t, tile_start, bucket_off, bucket_size, nbuckets, b, beg, c)) { d.bucket = b; d.begin = beg; d.count = c; }
    desc[t] = d;
}

__device__ __forceinline__ u32 smem_addr(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "WAIT_LOOP:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra WAIT_DONE;\n"
                 "bra WAIT_LOOP;\n"
                 "WAIT_DONE:\n"
                 "}" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy; dst, src and bytes are multiples of 16
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, u32 bytes, u64 *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

constexpr int QCE_MSDB_THREADS = 512, QCE_MSDB_ITEMS = 8;
constexpr int QCE_MSDB_SLOTS = QCE_MSD_TILE + 2;                 // a misaligned tile start costs up to 2 extra words
constexpr size_t QCE_MSDB_SMEM = 2 * QCE_MSDB_SLOTS * sizeof(u64); // dynamic shared memory of the kernel
// FROM_COL: `in` is a whole base column (keys below 2^32) and the tiles are those of one bucket
// covering it, so tile positions are row ids: the landed word w at position p is the tuple
// w << 32 | p.  The tuples are formed in registers and never stored unsorted (MSD level A straight
// from the column, qce_build_sorted_tuples_base).  The column's odd last word is loaded plainly
// rather than by a bulk copy reaching past its end.
template <bool FROM_COL> struct MsdbWord { using T = u64; };
template <> struct MsdbWord<true> { using T = u32; }; // a column word below 2^32: half the registers of a tuple
template <bool FROM_COL>
__global__ void __launch_bounds__(QCE_MSDB_THREADS, 3)
k_msd_partition_bulk(const u64 *__restrict__ in, u64 *__restrict__ out, const MsdTileDesc *__restrict__ desc, u32 ntiles,
                     u64 base, int shift, u32 bins, u32 *__restrict__ cursor)
{
    constexpr int THREADS = QCE_MSDB_THREADS, ITEMS = QCE_MSDB_ITEMS;
    extern __shared__ __align__(128) unsigned char msdb_smem[];
    u64 *const buf0 = reinterpret_cast<u64 *>(msdb_smem);
#define MSDB_BUF(b) (buf0 + (b) * QCE_MSDB_SLOTS)
    __shared__ __align__(8) u64 bar[2];
    __shared__ u32 cnt[256], excl[256], goff[256];
    __shared__ u32 scratch[33];
    __shared__ MsdTileDesc sdesc[2];
    const int tid = threadIdx.x;
    const u32 mask = bins - 1;

    // thread 0 is the producer: describe + fetch tile t into buffer b
    auto fetch = [&](u32 t, int b) {
        MsdTileDesc d = desc[t];
        sdesc[b] = d;
        if (d.count == 0) return;
        const u32 first = d.begin & ~1u, end = d.begin + d.count;
        u32 last = (end + 1u) & ~1u; // 16-byte aligned superset
        if (FROM_COL && (end & 1u)) {
            last = end - 1u;
            MSDB_BUF(b)[last - first] = in[last];
        }
        const u32 bytes = (last - first) * (u32)sizeof(u64);
        mbar_expect_tx(&bar[b], bytes);
        if (bytes) bulk_g2s(MSDB_BUF(b), in + first, bytes, &bar[b]);
    };
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 256) cnt[tid] = 0;
    __syncthreads();
    const u32 t0 = blockIdx.x, stride = gridDim.x;
    if (tid == 0) {
        if (t0 < ntiles) fetch(t0, 0);
        if (t0 + stride < ntiles) fetch(t0 + stride, 1);
    }
    __syncthreads();

    u32 it = 0;
    for (u32 t = t0; t < ntiles; t += stride, it++) {
        const int b = it & 1;
        const MsdTileDesc d = sdesc[b];
        const u32 count = d.count;
        typename MsdbWord<FROM_COL>::T key[ITEMS];
        u32 slot[ITEMS];
        if (count) {
            mbar_wait(&bar[b], (it >> 1) & 1);
            const u64 *src = MSDB_BUF(b) + (d.begin & 1u);
            bool agg = false;
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 i = tid + j * THREADS;
                const bool live = i < count;
                u32 dg = 0;
                if (live) {
                    key[j] = (typename MsdbWord<FROM_COL>::T)src[i];
                    const u64 k = FROM_COL ? (u64)key[j] << 32 : (u64)key[j]; // shift >= 32: the row id adds no digit bit
                    dg = (u32)((k - base) >> shift) & mask;
                }
                if (j == 0) agg = bins > 4 && msd_warp_skewed(dg, live);
                const u32 r = msd_rank(cnt, dg, live, agg);
                if (live) slot[j] = (dg << 16) | r;
            }
        }
        __syncthreads(); // every key of the tile is in registers: the buffer is free for staging
        {
            const u32 c = tid < 256 ? cnt[tid] : 0u;
            u32 tot;
            const u32 ex = block_scan_excl<u32, THREADS>(c, scratch, &tot);
            if (tid < 256) {
                excl[tid] = ex;
                goff[tid] = (c ? atomicAdd(&cursor[d.bucket * bins + tid], c) : 0u) - ex;
                cnt[tid] = 0; // for the next tile
            }
        }
        __syncthreads();
        u64 *stage = MSDB_BUF(b);
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 i = tid + j * THREADS;
            if (i < count)
                stage[excl[slot[j] >> 16] + (slot[j] & 0xffffu)] = FROM_COL ? ((u64)key[j] << 32) | (d.begin + i) : (u64)key[j];
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 p = tid + j * THREADS;
            if (p < count) {
                const u64 k = stage[p];
                out[goff[(u32)((k - base) >> shift) & mask] + p] = k;
            }
        }
        __syncthreads(); // staging reads done: the buffer may take the tile after next
        if (tid == 0 && t + 2 * stride < ntiles) {
            fence_proxy_async(); // generic-proxy writes to the buffer before the async-proxy copy into it
            fetch(t + 2 * stride, b);
        }
    }
#undef MSDB_BUF
}

// Largest segment length (to decide whether every sub-bucket fits the finish kernel).
// min and max of the per-tuple match counts of a merge (uniform multiplicity test, 8f-2)
__global__ void __launch_bounds__(256) k_minmax_u32(const u32 *__restrict__ v, u32 n, u32 *__restrict__ out_min, u32 *__restrict__ out_max)
{
    u32 lo = 0xffffffffu, hi = 0;
    for (u32 i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) { const u32 x = v[i]; lo = min(lo, x); hi = max(hi, x); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(QCE_FULL_MASK, lo, o));
        hi = max(hi, __shfl_xor_sync(QCE_FULL_MASK, hi, o));
    }
    if ((threadIdx.x & 31) == 0) { atomicMin(out_min, lo); atomicMax(out_max, hi); }
}
__global__ void __launch_bounds__(256) k_max_u32(const u32 *__restrict__ v, u32 n, u32 *__restrict__ out)
{
    u32 m = 0;
    for (u32 i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) m = max(m, v[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(QCE_FULL_MASK, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// Digit plan of the finish kernel: the remaining key bits split evenly over the
// passes (11 bits -> 6 + 5), so that no ballots are spent on bits that are zero.
struct LocalPlan {
    int npass;
    int shift[QCE_MAX_PASSES];
    int bits[QCE_MAX_PASSES];
};
__device__ __forceinline__ u32 warp_peers_dyn(u32 d, int bits)
{
    u32 peers = QCE_FULL_MASK;
    for (int b = 0; b < bits; b++) {
        asm("{\n\t"
            ".reg .pred p;\n\t"
            ".reg .b32 t, m, nm;\n\t"
            "and.b32 t, %1, %2;\n\t"
            "setp.ne.u32 p, t, 0;\n\t"
            "vote.sync.ballot.b32 m, p, 0xffffffff;\n\t"
            "selp.b32 nm, 0, 0xffffffff, p;\n\t"
            "lop3.b32 %0, %0, m, nm, 0x60;\n\t"
            "}"
            : "+r"(peers)
            : "r"(d), "r"(1u << b));
    }
    return peers;
}

// Finish: CTA s sorts segment s = [seg_off[s], seg_off[s] + seg_size[s]) in place
// on the planned digits (the key bits below the partition bits), all in shared
// memory.  Same ranking as k_block_sort; warps whose slots are all past the end
// of the segment skip the ranking work.  The host picks the smallest THREADS x
// ITEMS that holds the largest segment.
template <int THREADS, int ITEMS, int MIN_CTAS>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
k_msd_local_sort(u64 *__restrict__ keys, const u32 *__restrict__ seg_off, const u32 *__restrict__ seg_size,
                 u64 key_base, LocalPlan plan)
{
    constexpr int TILE = THREADS * ITEMS;
    constexpr int WARPS = THREADS / 32;
    constexpr int BINS = 256;
    __shared__ u64 skeys[TILE];
    __shared__ u32 warp_hist[WARPS * BINS];
    __shared__ u32 tile_excl[BINS];
    __shared__ u32 scratch[33];
    const u32 n = seg_size[blockIdx.x];
    if (n <= 1) return;
    u64 *base = keys + seg_off[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 lt = lanemask_lt();
    const u32 slot0 = warp * (32 * ITEMS) + lane;
    const bool warp_live = (u32)(warp * 32 * ITEMS) < n;

    u64 key[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 idx = slot0 + j * 32;
        key[j] = (idx < n) ? base[idx] : ~0ull;
    }
    for (int p = 0; p < plan.npass; p++) {
        const int shift = plan.shift[p], bits = plan.bits[p];
        const u32 mask = (1u << bits) - 1, nbins = 1u << bits;
        for (u32 i = tid; i < WARPS * BINS; i += THREADS) warp_hist[i] = 0;
        __syncthreads();
        u32 rd[ITEMS];
        u32 *wh = warp_hist + warp * BINS;
        if (warp_live) {
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 idx = slot0 + j * 32;
                // padding ranks behind every real tuple: top digit, and it comes last in run order
                const u32 d = (idx < n) ? ((u32)((key[j] - key_base) >> shift) & mask) : mask;
                const u32 peers = warp_peers_dyn(d, bits);
                u32 old = 0;
                if ((peers & lt) == 0) old = atomicAdd(&wh[d], (u32)__popc(peers));
                old = __shfl_sync(QCE_FULL_MASK, old, __ffs(peers) - 1);
                rd[j] = (d << 16) | (old + __popc(peers & lt));
            }
        }
        __syncthreads();
        u32 cnt = 0;
        if (tid < (int)nbins) {
#pragma unroll
            for (int w = 0; w < WARPS; w++) {
                const u32 c = warp_hist[w * BINS + tid];
                warp_hist[w * BINS + tid] = cnt;
                cnt += c;
            }
        }
        u32 tot;
        const u32 ex = block_scan_excl<u32, THREADS>(cnt, scratch, &tot);
        if (tid < BINS) tile_excl[tid] = ex;
        __syncthreads();
        if (warp_live) {
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 d = rd[j] >> 16;
                skeys[tile_excl[d] + wh[d] + (rd[j] & 0xffffu)] = key[j];
            }
        }
        __syncthreads();
        if (warp_live) {
#pragma unroll
            for (int j = 0; j < ITEMS; j++) key[j] = skeys[slot0 + j * 32];
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 idx = slot0 + j * 32;
        if (idx < n) base[idx] = key[j];
    }
}

// Finish, remaining bits R <= 12: one unstable counting sort per sub-bucket on ALL
// remaining key bits (2^R shared-memory counters).  Equal digits are now equal
// keys, so no stability is needed: a key's slot inside its digit comes from
// atomicAdd-with-return on the digit's counter -- no ballots, one pass.
// MAXB = counters cleared and scanned per sub-bucket (>= 2^rbits): with 11 remaining bits half of the
// 4096 is dead work that costs as much as ranking the ~2300 tuples themselves.
template <int THREADS, int ITEMS, int MIN_CTAS, int MAXB = 4096>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
k_msd_count_sort(u64 *__restrict__ keys, const u32 *__restrict__ seg_off, const u32 *__restrict__ seg_size,
                 u64 key_base, int rbits)
{
    constexpr int TILE = THREADS * ITEMS;
    constexpr int BPT = MAXB / THREADS; // counters per thread in the scan (consecutive)
    static_assert(BPT % 4 == 0, "the counter scan works on uint4 groups");
    extern __shared__ __align__(16) unsigned char smem_raw[]; // TILE*8 + MAXB*4 + 33*4 bytes
    u64 *skeys = reinterpret_cast<u64 *>(smem_raw);
    u32 *cnt = reinterpret_cast<u32 *>(skeys + TILE);
    u32 *scratch = cnt + MAXB;
    const u32 n = seg_size[blockIdx.x];
    if (n <= 1 || n > (u32)TILE) return; // oversized sub-buckets (a heavy key) take the k_big_* route
    u64 *base = keys + seg_off[blockIdx.x];
    const int tid = threadIdx.x;
    const u32 nb = 1u << rbits, mask = nb - 1;
    // all MAXB counters are cleared and scanned with 128-bit shared-memory accesses (a scalar
    // scan with `nb / THREADS` consecutive counters per thread is a 4- to 8-way bank conflict);
    // the counters beyond nb stay zero
    {
        uint4 *c4 = reinterpret_cast<uint4 *>(cnt);
#pragma unroll
        for (int q = 0; q < BPT / 4; q++) c4[tid + q * THREADS] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    u64 key[ITEMS];
    u32 slot[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < n) key[j] = base[i];
    }
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < n) slot[j] = atomicAdd(&cnt[(u32)((key[j] - key_base) >> 32) & mask], 1u);
    }
    __syncthreads();
    // exclusive scan of the counters in place (thread t owns BPT consecutive ones)
    {
        uint4 *c4 = reinterpret_cast<uint4 *>(cnt) + tid * (BPT / 4);
        uint4 v[BPT / 4];
        u32 sum = 0;
#pragma unroll
        for (int q = 0; q < BPT / 4; q++) {
            v[q] = c4[q];
            sum += v[q].x + v[q].y + v[q].z + v[q].w;
        }
        u32 tot;
        u32 ex = block_scan_excl<u32, THREADS>(sum, scratch, &tot);
#pragma unroll
        for (int q = 0; q < BPT / 4; q++) {
            uint4 o;
            o.x = ex; ex += v[q].x;
            o.y = ex; ex += v[q].y;
            o.z = ex; ex += v[q].z;
            o.w = ex; ex += v[q].w;
            c4[q] = o;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < n) skeys[cnt[(u32)((key[j] - key_base) >> 32) & mask] + slot[j]] = key[j];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < n) base[i] = skeys[i];
    }
}

// ---- the same finish with Blackwell-native data movement ------------------------------------------
// Persistent CTAs walk the sub-buckets; sub-bucket k+1 (and k+2) land in shared memory through the
// bulk-copy engine (cp.async.bulk + mbarrier, as in k_msd_partition_bulk) while sub-bucket k is counted,
// scanned and scattered -- the plain kernel above spends a third of every sub-bucket waiting for its own
// loads (ncu: long + short scoreboard, issue 27 %).  The landing buffer is the staging buffer.
template <int THREADS, int ITEMS, int MAXB>
__global__ void __launch_bounds__(THREADS, 3)
k_msd_count_sort_bulk(u64 *__restrict__ keys, const u32 *__restrict__ seg_off, const u32 *__restrict__ seg_size, u32 nsub,
                      u64 key_base, int rbits)
{
    constexpr int TILE = THREADS * ITEMS, SLOTS = TILE + 2;
    constexpr int BPT = MAXB / THREADS;
    static_assert(BPT % 4 == 0, "the counter scan works on uint4 groups");
    extern __shared__ __align__(128) unsigned char csb_smem[]; // 2 * SLOTS * 8 + MAXB * 4 bytes
    u64 *const buf0 = reinterpret_cast<u64 *>(csb_smem);
    u32 *const cnt = reinterpret_cast<u32 *>(buf0 + 2 * SLOTS);
    __shared__ __align__(8) u64 bar[2];
    __shared__ u32 scratch[33];
    __shared__ u32 sseg[2][2]; // offset, size of the sub-bucket in each buffer
    const int tid = threadIdx.x;
    const u32 nb = 1u << rbits, mask = nb - 1;
#define CSB_BUF(b) (buf0 + (b) * SLOTS)
    auto fetch = [&](u32 s, int b) {
        const u32 off = seg_off[s], n = seg_size[s];
        sseg[b][0] = off;
        sseg[b][1] = n > (u32)TILE ? 0u : n; // oversized sub-buckets (a heavy key) take the k_big_* route
        if (n <= 1 || n > (u32)TILE) return; // nothing to sort here, nothing to fetch
        const u32 first = off & ~1u, last = (off + n + 1u) & ~1u;
        const u32 bytes = (last - first) * (u32)sizeof(u64);
        mbar_expect_tx(&bar[b], bytes);
        bulk_g2s(CSB_BUF(b), keys + first, bytes, &bar[b]);
    };
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {
        uint4 *c4 = reinterpret_cast<uint4 *>(cnt);
#pragma unroll
        for (int q = 0; q < BPT / 4; q++) c4[tid + q * THREADS] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    const u32 s0 = blockIdx.x, stride = gridDim.x;
    if (tid == 0) {
        if (s0 < nsub) fetch(s0, 0);
        if (s0 + stride < nsub) fetch(s0 + stride, 1);
    }
    __syncthreads();
    u32 uses[2] = {0u, 0u}; // completed phases of each buffer's barrier (only sub-buckets with n > 1 use it)
    u32 it = 0;
    for (u32 s = s0; s < nsub; s += stride, it++) {
        const int b = it & 1;
        const u32 off = sseg[b][0], n = sseg[b][1];
        if (n > 1) {
            mbar_wait(&bar[b], uses[b] & 1u);
            uses[b]++;
            u64 key[ITEMS];
            u32 slot[ITEMS];
            const u64 *src = CSB_BUF(b) + (off & 1u);
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 i = tid + j * THREADS;
                if (i < n) {
                    key[j] = src[i];
                    slot[j] = atomicAdd(&cnt[(u32)((key[j] - key_base) >> 32) & mask], 1u);
                }
            }
            __syncthreads(); // keys in registers, counters complete
            {
                uint4 *c4 = reinterpret_cast<uint4 *>(cnt) + tid * (BPT / 4);
                uint4 v[BPT / 4];
                u32 sum = 0;
#pragma unroll
                for (int q = 0; q < BPT / 4; q++) {
                    v[q] = c4[q];
                    sum += v[q].x + v[q].y + v[q].z + v[q].w;
                }
                u32 tot;
                u32 ex = block_scan_excl<u32, THREADS>(sum, scratch, &tot);
#pragma unroll
                for (int q = 0; q < BPT / 4; q++) {
                    uint4 o;
                    o.x = ex; ex += v[q].x;
                    o.y = ex; ex += v[q].y;
                    o.z = ex; ex += v[q].z;
                    o.w = ex; ex += v[q].w;
                    c4[q] = o;
                }
            }
            __syncthreads();
            u64 *stage = CSB_BUF(b);
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 i = tid + j * THREADS;
                if (i < n) stage[cnt[(u32)((key[j] - key_base) >> 32) & mask] + slot[j]] = key[j];
            }
            __syncthreads();
            u64 *dst = keys + off;
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 i = tid + j * THREADS;
                if (i < n) dst[i] = stage[i];
            }
            {
                uint4 *c4 = reinterpret_cast<uint4 *>(cnt);
#pragma unroll
                for (int q = 0; q < BPT / 4; q++) c4[tid + q * THREADS] = make_uint4(0u, 0u, 0u, 0u);
            }
        }
        __syncthreads(); // staging reads done, counters clear: the buffer may take the sub-bucket after next
        if (tid == 0 && s + 2 * stride < nsub) {
            fence_proxy_async();
            fetch(s + 2 * stride, b);
        }
    }
#undef CSB_BUF
}

// ---- skew: sub-buckets a heavy key overflows ----------------------------------------------------------
// A sub-bucket larger than the finish kernel's tile (a key that alone has more than ~3000 tuples: config 4's
// Zipf side has ~1000 of them holding 78 % of the run) used to send the WHOLE run down four LSD passes.
// Only those sub-buckets now take another route: one more counting pass on ALL their remaining key bits
// (<= 12 bits -> <= 4096 bins, so equal digits are equal keys and nothing has to be stable): a
// multi-CTA histogram, a per-bucket scan, an unstable scatter into the ping-pong buffer, and a copy back.
// 40 B per tuple of the big sub-buckets instead of 72 B per tuple of everything.
__global__ void __launch_bounds__(256)
k_big_list(const u32 *__restrict__ sub_size, const u32 *__restrict__ sub_off, u32 nsub, u32 cap, u32 max_list,
           u32 *__restrict__ nbig, u32 *__restrict__ big_off, u32 *__restrict__ big_size, u32 *__restrict__ big_tiles)
{
    const u32 s = blockIdx.x * 256 + threadIdx.x;
    if (s >= nsub) return;
    const u32 n = sub_size[s];
    if (n <= cap) return;
    const u32 at = atomicAdd(nbig, 1u);
    if (at >= max_list) return; // the caller sees nbig > max_list and falls back
    big_off[at] = sub_off[s];
    big_size[at] = n;
    big_tiles[at] = (n + QCE_MSD_TILE - 1) / QCE_MSD_TILE;
}
__global__ void k_big_tile_total(u32 *__restrict__ tile_start, u32 nbig, const u64 *__restrict__ total)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) tile_start[nbig] = (u32)*total;
}
// ghist[bucket * nb + (low rbits of the key)] over the tiles of the big sub-buckets
template <int MAXB>
__global__ void __launch_bounds__(512)
k_big_hist(const u64 *__restrict__ keys, const MsdTileDesc *__restrict__ desc, u64 key_base, int rbits, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[MAXB];
    const MsdTileDesc d = desc[blockIdx.x];
    if (d.count == 0) return;
    const u32 nb = 1u << rbits, mask = nb - 1;
    for (u32 b = threadIdx.x; b < nb; b += 512) sh[b] = 0;
    __syncthreads();
    // a heavy key's tiles are one bin: warps whose lanes agree count once (32 atomics on one shared
    // address serialise)
    for (u32 i0 = (threadIdx.x & ~31u); i0 < d.count; i0 += 512) {
        const u32 i = i0 + (threadIdx.x & 31u);
        const bool valid = i < d.count;
        const u32 bin = valid ? (u32)((ld_stream_u64(keys + d.begin + i) - key_base) >> 32) & mask : 0xffffffffu;
        const u32 live = __ballot_sync(QCE_FULL_MASK, valid);
        const u32 first = __shfl_sync(QCE_FULL_MASK, bin, 0);
        if (__all_sync(QCE_FULL_MASK, bin == first || !valid)) {
            if ((threadIdx.x & 31u) == 0 && live) atomicAdd(&sh[first], (u32)__popc(live));
        } else if (valid) {
            atomicAdd(&sh[bin], 1u);
        }
    }
    __syncthreads();
    for (u32 b = threadIdx.x; b < nb; b += 512)
        if (sh[b]) atomicAdd(&ghist[(size_t)d.bucket * nb + b], sh[b]);
}
// in place: ghist[bucket][bin] -> exclusive prefix inside the bucket (one CTA per big sub-bucket)
__global__ void __launch_bounds__(1024) k_big_scan(u32 *__restrict__ ghist, u32 nb)
{
    __shared__ u32 scratch[33];
    u32 *h = ghist + (size_t)blockIdx.x * nb;
    u32 running = 0;
    for (u32 base = 0; base < nb; base += 1024) {
        const u32 b = base + threadIdx.x;
        const u32 v = b < nb ? h[b] : 0u;
        u32 tot;
        const u32 ex = block_scan_excl<u32, 1024>(v, scratch, &tot);
        if (b < nb) h[b] = running + ex;
        running += tot;
    }
}
// scatter the tiles of the big sub-buckets by the low rbits: out[bucket_off + cursor[bucket][bin]++]
template <int MAXB>
__global__ void __launch_bounds__(512, 2)
k_big_partition(const u64 *__restrict__ in, u64 *__restrict__ out, const MsdTileDesc *__restrict__ desc,
                const u32 *__restrict__ big_off, u64 key_base, int rbits, u32 *__restrict__ cursor)
{
    constexpr int THREADS = 512, ITEMS = QCE_MSD_TILE / THREADS;
    extern __shared__ __align__(16) unsigned char bigp_smem[]; // TILE * 8 + 3 * MAXB * 4 bytes
    u64 *skeys = reinterpret_cast<u64 *>(bigp_smem);
    u32 *cnt = reinterpret_cast<u32 *>(skeys + QCE_MSD_TILE), *excl = cnt + MAXB, *goff = excl + MAXB;
    __shared__ u32 scratch[33];
    const MsdTileDesc d = desc[blockIdx.x];
    if (d.count == 0) return;
    const int tid = threadIdx.x;
    const u32 nb = 1u << rbits, mask = nb - 1;
    for (u32 b = tid; b < nb; b += THREADS) cnt[b] = 0;
    __syncthreads();
    u64 key[ITEMS];
    u32 slot[ITEMS];
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS; // whole warps share `valid` except in the tail warp
        const bool valid = i < d.count;
        key[j] = valid ? ld_stream_u64(in + d.begin + i) : 0ull;
        const u32 bin = (u32)((key[j] - key_base) >> 32) & mask;
        const u32 live = __ballot_sync(QCE_FULL_MASK, valid);
        const u32 first = __shfl_sync(QCE_FULL_MASK, bin, __ffs(live) - 1 < 0 ? 0 : __ffs(live) - 1);
        if (__all_sync(QCE_FULL_MASK, !valid || bin == first)) {
            // the whole warp holds one key (a heavy hitter's tile): one shared atomic instead of 32 on one address
            u32 b0 = 0;
            if ((tid & 31) == 0 && live) b0 = atomicAdd(&cnt[first], (u32)__popc(live));
            b0 = __shfl_sync(QCE_FULL_MASK, b0, 0);
            slot[j] = b0 + (u32)__popc(live & lt);
        } else if (valid) {
            slot[j] = atomicAdd(&cnt[bin], 1u);
        }
    }
    __syncthreads();
    // exclusive scan of the tile's counters (MAXB / THREADS consecutive ones per thread) and the
    // reservation of the tile's output range per populated bin
    {
        constexpr int BPT = MAXB / THREADS;
        u32 v[BPT], sum = 0;
#pragma unroll
        for (int q = 0; q < BPT; q++) {
            const u32 b = tid * BPT + q;
            v[q] = b < nb ? cnt[b] : 0u;
            sum += v[q];
        }
        u32 tot;
        u32 ex = block_scan_excl<u32, THREADS>(sum, scratch, &tot);
#pragma unroll
        for (int q = 0; q < BPT; q++) {
            const u32 b = tid * BPT + q;
            if (b < nb) {
                excl[b] = ex;
                goff[b] = (v[q] ? atomicAdd(&cursor[(size_t)d.bucket * nb + b], v[q]) : 0u) - ex;
            }
            ex += v[q];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < d.count) skeys[excl[(u32)((key[j] - key_base) >> 32) & mask] + slot[j]] = key[j];
    }
    __syncthreads();
    u64 *dst = out + big_off[d.bucket];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 p = tid + j * THREADS;
        if (p < d.count) {
            const u64 k = skeys[p];
            dst[goff[(u32)((k - key_base) >> 32) & mask] + p] = k;
        }
    }
}
__global__ void __launch_bounds__(512)
k_big_copyback(const u64 *__restrict__ from, u64 *__restrict__ to, const MsdTileDesc *__restrict__ desc)
{
    const MsdTileDesc d = desc[blockIdx.x];
    for (u32 i = threadIdx.x; i < d.count; i += 512) to[d.begin + i] = ld_stream_u64(from + d.begin + i);
}

// 1 if keys[i-1] > keys[i] anywhere (checks the "already sorted" assumption of
// JOIN_SORT_LHS / JOIN_SORT_RHS, src/join.c:647-658).
template <bool WIDE>
__global__ void __launch_bounds__(256) k_is_unsorted(TupleView t, u64 n, u32 *__restrict__ flag)
{
    const u64 stride = (u64)gridDim.x * 256;
    bool bad = false;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x + 1; i < n; i += stride)
        bad |= tv_key<WIDE>(t, i - 1) > tv_key<WIDE>(t, i);
    if (__any_sync(QCE_FULL_MASK, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}
