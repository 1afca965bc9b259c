// k_exchange.cuh -- partition + push over NVLink peer memory (SURVEY.md 8e).
//
// The reference has no exchange step (one process, one thread); this is the
// multi-GPU half of its radix partitioning (build_histogram / build_psum /
// build_reordered_array, src/utilities.c:20-70): the scatter pass of the top
// radix digit writes every tuple straight into the receive window of the GPU
// that owns its key range.  One kernel does the partition AND the transfer:
// a 4096-tuple tile is grouped by destination in shared memory and each group
// leaves as one coalesced run of stores -- into local HBM for the rank's own
// share, over NVLink (P2P stores through an IPC-mapped window) for the others.
// Nothing is staged in a send buffer and there is no separate all-to-all.
//
// Offsets are deterministic: every rank holds the all-gathered 256-bin
// histograms of all ranks, so it knows where its segment starts inside every
// destination window before the kernel is launched; the only device-side
// coordination is one 64-bit atomicAdd per (tile, destination) on a LOCAL cursor.
//
// Two element types:
//   * packed tuples (key << 32 | payload), destination = table[top 8 key bits];
//     optionally the payload is replaced by the tuple's index in the receiver's
//     run and the tuple's slot is recorded, so that bystander row-id columns of
//     the same entity can follow it (k_push_u32_by_slot);
//   * 4-byte row ids, digit = id / bin_width (<= 256 equal-width bins of the
//     relation's row domain), destination = the rank that owns the bin's rows.
//     The receiver gets its ids grouped by bin, i.e. already bucketed for
//     L2-resident checksum gathers (this replaces partition_ids_by_top_bits);
//   * wide runs (SoA u64 keys + u32 ids, k_push_wide): destination = table[top 8
//     bits of key - base], the ids follow the keys through the same staged tile.
//
// Algorithmic bytes: 8 B read + 8 B written per tuple (4 + 4 per id); the
// written bytes cross NVLink for the (G-1)/G share that leaves the rank.
#pragma once
#include "k_radix.cuh"

#define QCE_PUSH_THREADS 512
// 32 KB of shared-memory staging per tile: 4096 tuples, or 8192 row ids (a 256-bin id
// scatter then leaves in runs of ~32 ids = 128 B, the NVLink write granularity that pays)
template <typename KeyT> struct PushTile { static constexpr int ITEMS = sizeof(KeyT) == 8 ? 8 : 16; static constexpr int TILE = QCE_PUSH_THREADS * ITEMS; };

struct PeerWindows {
    unsigned char *base[QCE_MAX_RANKS]; // receive window of every rank, mapped into this process
};

struct PushPlan {
    const unsigned long long *seg_start; // [ndigits] element offset of this rank's segment in the owner's window
    const u32 *run_base;                 // [ndigits] index of that segment's first element in the receiver's run
    unsigned long long *cursor;          // [ndigits] next free element offset (starts at seg_start), LOCAL memory
    u32 ndigits;
    u32 digits_per_rank;                 // owner rank of digit d = d / digits_per_rank
};

template <typename KeyT> struct PushDigit;
// tuples: 256-bin histogram digit of the key -> destination rank through a byte table
template <> struct PushDigit<u64> {
    int shift;
    const u32 *lut; // 256 bytes packed in 64 words
    __device__ __forceinline__ u32 operator()(u64 w) const
    {
        const u32 b = (u32)(w >> shift) & 255u;
        return (__ldg(lut + (b >> 2)) >> ((b & 3u) * 8)) & 255u;
    }
};
// row ids: owner rank = id / rows_per_rank, then equal-width bins inside the owner's rows
struct RowBins {
    u32 rows_per_rank, last_rank, width, bins_per_rank;
    float inv_rows; // 1 / rows_per_rank, rounded down
    __host__ __device__ __forceinline__ u32 operator()(u32 id) const
    {
        if (bins_per_rank == 1) { // owner only: reciprocal multiply + one-step correction (no division)
#ifdef __CUDA_ARCH__
            u32 r = min(__float2uint_rz(__uint2float_rz(id) * inv_rows), last_rank);
            r -= (id < r * rows_per_rank);
            r += (r < last_rank) & (id >= (r + 1) * rows_per_rank);
            return r;
#else
            return id / rows_per_rank < last_rank ? id / rows_per_rank : last_rank;
#endif
        }
        const u32 r = min(id / rows_per_rank, last_rank);
        return r * bins_per_rank + min((id - r * rows_per_rank) / width, bins_per_rank - 1);
    }
};
template <> struct PushDigit<u32> {
    RowBins bins;
    __device__ __forceinline__ u32 operator()(u32 id) const { return bins(id); }
};

// Bystander columns that travel with a run: column c of input tuple i is stored at 4-byte
// element region[c][d] + (position of the tuple inside this rank's segment of destination d),
// i.e. at the tuple's index in the receiver's run when the regions are laid out like the runs.
#define QCE_PUSH_MAX_COLS 6
struct PushCols {
    const u32 *in[QCE_PUSH_MAX_COLS];
    unsigned long long region[QCE_PUSH_MAX_COLS][QCE_MAX_RANKS];
    int n;
};

// FEW: at most 16 digits -> ranks inside the tile come from per-bit ballots and
// one shared atomicAdd per (warp, digit) group; otherwise one shared atomicAdd
// per element (256 digits, little contention).
template <typename KeyT, bool FEW, bool REWRITE>
__global__ void __launch_bounds__(QCE_PUSH_THREADS, sizeof(KeyT) == 8 ? 3 : 2)
k_push(const KeyT *__restrict__ in, u32 n, PushDigit<KeyT> digit, PushPlan plan, const __grid_constant__ PeerWindows peers, int digit_bits,
       u32 *__restrict__ slot_out, const __grid_constant__ PushCols cols)
{
    constexpr int THREADS = QCE_PUSH_THREADS, ITEMS = PushTile<KeyT>::ITEMS, TILE = PushTile<KeyT>::TILE;
    __shared__ KeyT skeys[TILE];
    __shared__ unsigned char sdig[TILE]; // digit of the element staged at each tile position
    __shared__ u32 cnt[256], excl[256];
    __shared__ unsigned long long goff[256]; // reserved start of the tile's run in the window, minus excl
    __shared__ unsigned long long sseg[256];
    __shared__ u32 srun[256];
    __shared__ u32 scratch[33];
    const int tid = threadIdx.x, lane = tid & 31;
    const u32 begin = blockIdx.x * TILE;
    if (begin >= n) return;
    const u32 count = min((u32)TILE, n - begin);
    if (tid < 256) cnt[tid] = 0;
    __syncthreads();

    KeyT key[ITEMS];
    u32 slot[ITEMS]; // digit << 16 | rank among the tile's elements with that digit
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        key[j] = (i < count) ? ld_stream_key<KeyT>(in + begin + i) : (KeyT)0;
    }
    if (FEW) {
        // cnt[d * 16 + warp]: every warp counts its own elements per digit, so nothing is
        // contended (one shared atomicAdd per warp-group on 2-16 addresses serialised the
        // whole tile: 2.6x slower than the memory traffic).  The 256-entry scan below then
        // yields, per (digit, warp), where that warp's elements start inside the tile.
        const u32 lt = lanemask_lt();
        const u32 warp = tid >> 5;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 i = tid + j * THREADS;
            const bool valid = i < count; // whole warps share `valid` except in the tail warp
            const u32 d = valid ? digit(key[j]) : 0u;
            const u32 live = __ballot_sync(QCE_FULL_MASK, valid);
            const u32 peersm = warp_peers_dyn(d, digit_bits) & live;
            u32 b = 0;
            const int leader = __ffs(peersm) - 1;
            if (valid && lane == leader) {
                b = cnt[d * 16 + warp];
                cnt[d * 16 + warp] = b + (u32)__popc(peersm);
            }
            __syncwarp();
            b = __shfl_sync(QCE_FULL_MASK, b, leader < 0 ? 0 : leader);
            slot[j] = (d << 16) | (b + (u32)__popc(peersm & lt));
        }
    } else {
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 i = tid + j * THREADS;
            if (i < count) {
                const u32 d = digit(key[j]);
                slot[j] = (d << 16) | atomicAdd(&cnt[d], 1u);
            }
        }
    }
    __syncthreads();
    {
        const u32 c = (tid < 256) ? cnt[tid] : 0u;
        u32 tot;
        const u32 ex = block_scan_excl<u32, THREADS>(c, scratch, &tot);
        if (tid < 256) excl[tid] = ex;
        if (FEW) {
            __syncthreads();
            if (tid < plan.ndigits) {
                // digit tid: elements of all 16 warps
                const u32 first = excl[tid * 16], end = (tid + 1 < 16) ? excl[(tid + 1) * 16] : tot;
                const u32 cd = end - first;
                unsigned long long r = 0;
                if (cd) r = atomicAdd(&plan.cursor[tid], (unsigned long long)cd);
                goff[tid] = r - first;
            }
        } else if (tid < 256) {
            unsigned long long r = 0;
            if (c) r = atomicAdd(&plan.cursor[tid], (unsigned long long)c);
            goff[tid] = r - ex;
        }
        if (tid < plan.ndigits) { sseg[tid] = plan.seg_start[tid]; srun[tid] = plan.run_base[tid]; }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < count) {
            const u32 d = slot[j] >> 16, p = excl[FEW ? d * 16 + (tid >> 5) : d] + (slot[j] & 0xffffu);
            skeys[p] = key[j];
            sdig[p] = (unsigned char)d;
            slot[j] = p; // from here on: the element's position in the staged tile
            // where the element lands, relative to this rank's segment in the owner's window
            if (slot_out) slot_out[begin + i] = (d << 28) | (u32)(goff[d] + p - sseg[d]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 p = tid + j * THREADS;
        if (p < count) {
            KeyT k = skeys[p];
            const u32 d = sdig[p];
            const unsigned long long at = goff[d] + p;
            if (REWRITE) k = (KeyT)((k & ~(KeyT)0xffffffffu) | (KeyT)(srun[d] + (u32)(at - sseg[d])));
            ((KeyT *)peers.base[d / plan.digits_per_rank])[at] = k;
        }
    }
    if (REWRITE) {
        // the run's bystander columns, staged through the same tile order so that they too
        // leave as one coalesced run per destination (a 4-byte scatter by slot over NVLink
        // measured 11 ms for three joins of config 3 on 8 GPUs)
        u32 *scol = reinterpret_cast<u32 *>(skeys);
        for (int c = 0; c < cols.n; c++) {
            __syncthreads(); // everyone is done reading the previous contents of the staging buffer
            const u32 *__restrict__ src = cols.in[c] + begin;
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 i = tid + j * THREADS;
                if (i < count) scol[slot[j]] = ld_stream_u32(src + i);
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const u32 p = tid + j * THREADS;
                if (p < count) {
                    const u32 d = sdig[p];
                    ((u32 *)peers.base[d])[cols.region[c][d] + (goff[d] + p - sseg[d])] = scol[p];
                }
            }
        }
    }
}

// Wide runs (keys >= 2^32: SoA u64 keys + u32 row ids).  Such keys usually sit at a high offset
// (64-bit ids, timestamps), so the digit is the top byte of key - base over the exchange's width,
// not of the key itself: the top bits of the key would put every tuple in one bin.
struct PushDigitWide {
    u64 base;
    int shift; // width - 8 (0 below 8 bits)
    const u32 *lut;
    __device__ __forceinline__ u32 operator()(u64 k) const
    {
        const u32 b = (u32)((k - base) >> shift) & 255u;
        return (__ldg(lut + (b >> 2)) >> ((b & 3u) * 8)) & 255u;
    }
};
// id of the key stored at word w of destination d's window goes to 4-byte element w + id_delta[d]
// (the id region is laid out like the key region; the delta wraps mod 2^64 when it is "negative")
struct WideIdRegions {
    unsigned long long id_delta[QCE_MAX_RANKS];
};

// k_push<u64, FEW, false> for a wide run: the key word leaves unchanged, and the row id is staged
// through the same tile order (the REWRITE columns' mechanism) so that it too leaves as one
// coalesced run per destination.  Destinations <= 16 (per-warp ballot ranking).
__global__ void __launch_bounds__(QCE_PUSH_THREADS, 3)
k_push_wide(const u64 *__restrict__ keys, const u32 *__restrict__ ids, u32 n, PushDigitWide digit, PushPlan plan,
            const __grid_constant__ PeerWindows peers, int digit_bits, const __grid_constant__ WideIdRegions idr)
{
    constexpr int THREADS = QCE_PUSH_THREADS, ITEMS = PushTile<u64>::ITEMS, TILE = PushTile<u64>::TILE;
    __shared__ u64 skeys[TILE];
    __shared__ unsigned char sdig[TILE];
    __shared__ u32 cnt[256], excl[256];
    __shared__ unsigned long long goff[256];
    __shared__ u32 scratch[33];
    const int tid = threadIdx.x, lane = tid & 31;
    const u32 begin = blockIdx.x * TILE;
    if (begin >= n) return;
    const u32 count = min((u32)TILE, n - begin);
    if (tid < 256) cnt[tid] = 0;
    __syncthreads();

    // the keys wait in shared memory (input order) while they are ranked, and only their destinations
    // (4 bits each) stay in registers: holding eight keys through the ranking spills at 3 CTAs per SM
    u32 dest = 0;
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < count) {
            const u64 k = ld_stream_u64(keys + begin + i);
            skeys[i] = k;
            dest |= digit(k) << (4 * j);
        }
    }
    u32 slot[ITEMS]; // digit << 16 | rank among the tile's elements with that digit
    {
        // cnt[d * 16 + warp], as in k_push<FEW>
        const u32 lt = lanemask_lt();
        const u32 warp = tid >> 5;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const u32 i = tid + j * THREADS;
            const bool valid = i < count;
            const u32 d = (dest >> (4 * j)) & 15u;
            const u32 live = __ballot_sync(QCE_FULL_MASK, valid);
            const u32 peersm = warp_peers_dyn(d, digit_bits) & live;
            u32 b = 0;
            const int leader = __ffs(peersm) - 1;
            if (valid && lane == leader) {
                b = cnt[d * 16 + warp];
                cnt[d * 16 + warp] = b + (u32)__popc(peersm);
            }
            __syncwarp();
            b = __shfl_sync(QCE_FULL_MASK, b, leader < 0 ? 0 : leader);
            slot[j] = (d << 16) | (b + (u32)__popc(peersm & lt));
        }
    }
    __syncthreads();
    {
        const u32 c = (tid < 256) ? cnt[tid] : 0u;
        u32 tot;
        const u32 ex = block_scan_excl<u32, THREADS>(c, scratch, &tot);
        if (tid < 256) excl[tid] = ex;
        __syncthreads();
        if (tid < plan.ndigits) {
            const u32 first = excl[tid * 16], end = (tid + 1 < 16) ? excl[(tid + 1) * 16] : tot;
            const u32 cd = end - first;
            unsigned long long r = 0;
            if (cd) r = atomicAdd(&plan.cursor[tid], (unsigned long long)cd);
            goff[tid] = r - first;
        }
    }
    u64 key[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        key[j] = (i < count) ? skeys[i] : 0ull;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < count) {
            const u32 d = slot[j] >> 16, p = excl[d * 16 + (tid >> 5)] + (slot[j] & 0xffffu);
            skeys[p] = key[j];
            sdig[p] = (unsigned char)d;
            slot[j] = p;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 p = tid + j * THREADS;
        if (p < count) {
            const u32 d = sdig[p];
            ((u64 *)peers.base[d])[goff[d] + p] = skeys[p];
        }
    }
    __syncthreads(); // the staging buffer takes the ids now
    u32 *sids = reinterpret_cast<u32 *>(skeys);
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 i = tid + j * THREADS;
        if (i < count) sids[slot[j]] = ld_stream_u32(ids + begin + i);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u32 p = tid + j * THREADS;
        if (p < count) {
            const u32 d = sdig[p];
            ((u32 *)peers.base[d])[goff[d] + p + idr.id_delta[d]] = sids[p];
        }
    }
}

// 256-bin histogram of (key - base) >> shift over a wide run (the counts every rank all-gathers
// before k_push_wide)
__global__ void __launch_bounds__(512)
k_hist_wide(const u64 *__restrict__ keys, u64 n, u64 base, int shift, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[256];
    if (threadIdx.x < 256) sh[threadIdx.x] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * 1024;
    for (u64 e = ((u64)blockIdx.x * 512 + threadIdx.x) * 2; e < n; e += stride) {
        if (e + 1 < n) {
            u64 a, b;
            ld_stream_u64x2(keys + e, a, b);
            atomicAdd(&sh[(u32)((a - base) >> shift) & 255u], 1u);
            atomicAdd(&sh[(u32)((b - base) >> shift) & 255u], 1u);
        } else {
            atomicAdd(&sh[(u32)((keys[e] - base) >> shift) & 255u], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x < 256 && sh[threadIdx.x]) atomicAdd(&ghist[threadIdx.x], sh[threadIdx.x]);
}

// out[0] = max(~w), out[1] = max(w) over n words (out zeroed first): the smallest and largest word
// in the form the ranks' all-reduce (a max) combines
__global__ void __launch_bounds__(256)
k_minmax_u64(const u64 *__restrict__ w, u64 n, unsigned long long *__restrict__ out)
{
    u64 lo = ~0ull, hi = 0;
    const u64 stride = (u64)gridDim.x * 512;
    for (u64 e = ((u64)blockIdx.x * 256 + threadIdx.x) * 2; e < n; e += stride) {
        if (e + 1 < n) {
            u64 a, b;
            ld_stream_u64x2(w + e, a, b);
            lo = min(lo, min(a, b));
            hi = max(hi, max(a, b));
        } else {
            lo = min(lo, w[e]);
            hi = max(hi, w[e]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(QCE_FULL_MASK, lo, o));
        hi = max(hi, __shfl_xor_sync(QCE_FULL_MASK, hi, o));
    }
    if ((threadIdx.x & 31) == 0) { atomicMax(out, ~lo); atomicMax(out + 1, hi); }
}

// A packed run widened for a wide exchange: keys[i] = in[i] >> 32, ids[i] = (u32)in[i]
__global__ void __launch_bounds__(256)
k_unpack_wide(const u64 *__restrict__ in, u64 n, u64 *__restrict__ keys, u32 *__restrict__ ids)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const u64 w = ld_stream_u64(in + i);
        keys[i] = w >> 32;
        ids[i] = (u32)w;
    }
}

// Bystander column of a pushed entity: vals[i] goes where tuple i went
// (slot = destination << 28 | offset inside this rank's segment); region[d] is
// the u32 element offset of the matching segment in destination d's window.
struct SlotRegions {
    unsigned long long region[QCE_MAX_RANKS];
};
__global__ void __launch_bounds__(256)
k_push_u32_by_slot(const u32 *__restrict__ vals, const u32 *__restrict__ slot, u64 n, const __grid_constant__ SlotRegions reg,
                   const __grid_constant__ PeerWindows peers)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const u32 s = ld_stream_u32(slot + i);
        const u32 d = s >> 28;
        ((u32 *)peers.base[d])[reg.region[d] + (s & 0x0fffffffu)] = ld_stream_u32(vals + i);
    }
}

// 256-bin histogram of row ids over equal-width bins (the counts every rank
// all-gathers before k_push<u32>).
template <int NB> // NB = 2, 4, 8, 16: register counters for nbins <= NB; 256: shared atomics
__global__ void __launch_bounds__(512)
k_hist_u32_div(const u32 *__restrict__ ids, u64 n, RowBins bins, u32 nbins, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[256];
    if (threadIdx.x < 256) sh[threadIdx.x] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * 512;
    if (NB <= 16) {
        // few bins (one per owner rank): shared atomics on 2-16 addresses would serialise;
        // count in registers, reduce per warp at the end
        u32 c[NB <= 16 ? NB : 1];
#pragma unroll
        for (int k = 0; k < (NB <= 16 ? NB : 1); k++) c[k] = 0;
        const u64 n4 = n & ~3ull; // 128-bit loads, two in flight per thread
        for (u64 e = ((u64)blockIdx.x * 512 + threadIdx.x) * 4; e < n4; e += stride * 8) {
            const uint4 a = ld_stream_u32x4(ids + e);
            const bool two = e + stride * 4 < n4;
            const uint4 b4 = two ? ld_stream_u32x4(ids + e + stride * 4) : make_uint4(0, 0, 0, 0);
            const u32 v[8] = {a.x, a.y, a.z, a.w, b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (q >= 4 && !two) break;
                const u32 b = bins(v[q]);
#pragma unroll
                for (int k = 0; k < (NB <= 16 ? NB : 1); k++) c[k] += (b == (u32)k);
            }
        }
        if (blockIdx.x == 0 && threadIdx.x < n - n4) {
            const u32 b = bins(ids[n4 + threadIdx.x]);
#pragma unroll
            for (int k = 0; k < (NB <= 16 ? NB : 1); k++) c[k] += (b == (u32)k);
        }
#pragma unroll
        for (int k = 0; k < (NB <= 16 ? NB : 1); k++) {
            const u32 w = warp_sum_u32(c[k]);
            if ((threadIdx.x & 31) == 0 && w) atomicAdd(&sh[k], w);
        }
    } else {
        for (u64 i = (u64)blockIdx.x * 512 + threadIdx.x; i < n; i += stride)
            atomicAdd(&sh[bins(ld_stream_u32(ids + i))], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 256 && sh[threadIdx.x]) atomicAdd(&ghist[threadIdx.x], sh[threadIdx.x]);
}

// out[i] = src[index[i]] (bystander row ids re-aligned with a join output).
__global__ void __launch_bounds__(256)
k_gather_u32(const u32 *__restrict__ src, const u32 *__restrict__ index, u64 n, u32 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) out[i] = __ldg(src + ld_stream_u32(index + i));
}

// Carried join-key column: the low 32 bits of rows [begin, begin + n) of a base column.
__global__ void __launch_bounds__(256)
k_narrow_u64(const u64 *__restrict__ col, u64 n, u32 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) out[i] = (u32)ld_stream_u64(col + i);
}
__global__ void __launch_bounds__(256) k_iota_u32(u32 begin, u64 n, u32 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) out[i] = begin + (u32)i;
}
// Packed run over a carried key column: out[i] = keys[i] << 32 | i.
__global__ void __launch_bounds__(256)
k_pack_u32_index(const u32 *__restrict__ keys, u64 n, u64 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) out[i] = ((u64)ld_stream_u32(keys + i) << 32) | i;
}
// Carried key column through a row-id column: out[i] = (u32)col[ids[i]].
__global__ void __launch_bounds__(256)
k_gather_u64_narrow(const __grid_constant__ ColRef col, const u32 *__restrict__ ids, u64 n, u32 *__restrict__ out)
{
    const u64 stride = (u64)gridDim.x * 256;
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) out[i] = (u32)col(ld_stream_u32(ids + i));
}
