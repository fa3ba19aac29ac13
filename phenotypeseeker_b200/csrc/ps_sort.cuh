// ps_sort.cuh — hand-written stable LSD radix sort (one-sweep, decoupled look-back) for
// (k-mer key [, u16 sample tag]) pairs, plus the small scan / run-length kernels around it.
//
// Replaces the counting core of `glistmaker` and the merge passes of `glistcompare -u`
// (modeling.py:303-315, 351-380): k-mer instances of ALL samples are sorted once; equal
// k-mers end up adjacent, in sample order because the sort is stable.
//
// One pass = one read + one write of every pair: a tile of 4096 pairs is ranked in shared
// memory (warp-private digit histograms; lanes with equal digits meet through one shared
// atomicOr on a per-warp mask word), tiles chain their per-digit prefixes through a 64-bit status|value look-back
// word, and the tile is written out digit-run by digit-run (coalesced).
#pragma once
#include "ps_common.cuh"

#ifndef RS_THREADS
#define RS_THREADS 512
#endif
#ifndef RS_ITEMS
#define RS_ITEMS 16
#endif
#define RS_WARPS (RS_THREADS / 32)
#define RS_TILE (RS_THREADS * RS_ITEMS)  // 4096
#define RS_RADIX 256          // 8-bit digits (default)
#define RS_MAX_RADIX 512      // 9-bit digits: used when they save a whole pass (e.g. k = 13: 26 bits)
#define RS_MAX_PASSES 8
#ifndef RS_MIN_BLOCKS
#define RS_MIN_BLOCKS (1024 / RS_THREADS)
#endif
#ifndef RS_LB_BATCH
#define RS_LB_BATCH 4
#endif
#ifndef RS_RANK_ATOMIC
#define RS_RANK_ATOMIC 0
#endif
#ifndef RS_MATCH_BALLOT
#define RS_MATCH_BALLOT 1
#endif

template <typename KeyT, bool HAS_VAL> constexpr size_t rs_dyn_smem() {
    return RS_TILE * sizeof(KeyT) + (HAS_VAL ? RS_TILE * 2 : 0);
}

#define LB_LOCAL (1ull << 62)
#define LB_INCL (2ull << 62)
#define LB_MASK ((1ull << 62) - 1)

// Digit histograms of every pass in one read of the keys.
template <typename KeyT>
__global__ void __launch_bounds__(512)
k_rs_hist(const KeyT *__restrict__ keys, uint64_t n, int npass, int shift0, int rb,
          unsigned long long *__restrict__ hist) {
    __shared__ uint32_t sh[RS_MAX_PASSES][RS_MAX_RADIX];
    const uint32_t dmask = (1u << rb) - 1u;
    for (int i = threadIdx.x; i < RS_MAX_PASSES * RS_MAX_RADIX; i += blockDim.x) (&sh[0][0])[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        KeyT key = keys[i];
        for (int p = 0; p < npass; p++) atomicAdd(&sh[p][(uint32_t)(key >> (shift0 + rb * p)) & dmask], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < npass * RS_MAX_RADIX; i += blockDim.x) {
        uint32_t v = (&sh[0][0])[i];
        if (v) atomicAdd(&hist[i], (unsigned long long)v);
    }
}

// Exclusive scan of each pass's 256 bins: one block per pass.
__global__ void k_rs_scan(unsigned long long *__restrict__ hist) {
    __shared__ unsigned long long s[RS_MAX_RADIX];
    unsigned long long *h = hist + (size_t)blockIdx.x * RS_MAX_RADIX;
    s[threadIdx.x] = h[threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int i = 0; i < RS_MAX_RADIX; i++) { unsigned long long c = s[i]; s[i] = run; run += c; }
    }
    __syncthreads();
    h[threadIdx.x] = s[threadIdx.x];
}

template <typename KeyT, bool HAS_VAL, int RB>
__global__ void __launch_bounds__(RS_THREADS, ((sizeof(KeyT) == 8 && HAS_VAL && RS_MIN_BLOCKS > 1) ? RS_MIN_BLOCKS - 1 : RS_MIN_BLOCKS))
k_rs_pass(const KeyT *__restrict__ kin, KeyT *__restrict__ kout, const uint16_t *__restrict__ vin,
          uint16_t *__restrict__ vout, uint64_t n, int shift,
          const unsigned long long *__restrict__ gbase, unsigned long long *lookback,
          uint32_t *tile_counter) {
    constexpr int RADIX = 1 << RB;
    static_assert(RADIX <= RS_THREADS, "every digit needs an owner thread");
    __shared__ uint32_t whist[RS_WARPS][RADIX];  // per-warp digit counts, later scatter bases
    __shared__ uint32_t wmask[RS_WARPS][RADIX];  // per-warp lane mask per digit (self-clearing)
    extern __shared__ __align__(16) uint8_t rs_dyn[];  // RS_TILE keys, then RS_TILE u16 tags
    KeyT *skeys = reinterpret_cast<KeyT *>(rs_dyn);
    uint16_t *svals = reinterpret_cast<uint16_t *>(rs_dyn + RS_TILE * sizeof(KeyT));
    __shared__ unsigned long long goff[RADIX];
    __shared__ uint32_t wsum[RS_WARPS];
    __shared__ uint32_t s_tile;

    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
    for (int i = tid; i < RS_WARPS * RADIX; i += RS_THREADS) {
        (&whist[0][0])[i] = 0;
        (&wmask[0][0])[i] = 0;
    }
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t tile_start = (uint64_t)tile * RS_TILE;
    const uint32_t nvalid = (uint32_t)min((uint64_t)RS_TILE, n - tile_start);

    // warp-striped load: stable order inside the tile is (warp, item, lane)
    KeyT key[RS_ITEMS];
    uint16_t rank[RS_ITEMS];
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t idx = warp * (32 * RS_ITEMS) + i * 32 + lane;
        key[i] = idx < nvalid ? kin[tile_start + idx] : ~KeyT(0);
    }
    // Stable ranking inside the warp. Lanes holding the same digit find each other through
    // one shared-memory atomicOr on a per-warp mask word (MATCH.ANY costs ~one step per
    // distinct value and was the top stall of the first version of this kernel); the lowest
    // lane of each group bumps the warp-private digit counter and clears the mask.
    uint32_t *wh = whist[warp], *wm = wmask[warp];
    const unsigned lt = lanemask_lt();
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t d = (uint32_t)(key[i] >> shift) & (uint32_t)(RADIX - 1);
#if RS_RANK_ATOMIC
        rank[i] = (uint16_t)atomicAdd(wh + d, 1u);
#elif RS_MATCH_BALLOT
        // peers = lanes with the same digit: one ballot per digit bit, no shared memory
        unsigned peers = 0xffffffffu;
#pragma unroll
        for (int b = 0; b < RB; b++) {
            const bool bit = (d >> b) & 1u;
            const unsigned bal = __ballot_sync(0xffffffffu, bit);
            peers &= bit ? bal : ~bal;
        }
        const uint32_t old = wh[d];
        __syncwarp();
        const uint32_t r = __popc(peers & lt);
        if (r == 0) wh[d] = old + __popc(peers);
        rank[i] = (uint16_t)(old + r);
        __syncwarp();
#else
        atomicOr(wm + d, 1u << lane);
        __syncwarp();
        const unsigned peers = wm[d];
        const uint32_t old = wh[d];
        __syncwarp();
        const uint32_t r = __popc(peers & lt);
        if (r == 0) {
            wh[d] = old + __popc(peers);
            wm[d] = 0;
        }
        rank[i] = (uint16_t)(old + r);
        __syncwarp();
#endif
    }
    // tags: issue the loads now, their latency hides behind the scan + look-back
    uint16_t val[HAS_VAL ? RS_ITEMS : 1];
    if (HAS_VAL) {
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) {
            const uint32_t idx = warp * (32 * RS_ITEMS) + i * 32 + lane;
            val[i] = idx < nvalid ? vin[tile_start + idx] : (uint16_t)0;
        }
    }

    __syncthreads();   // every warp finished ranking, whist is final

    // digit `tid`: tile count, published at once as this tile's LOCAL look-back entry
    const bool dig = tid < RADIX;   // threads that own a digit
    uint32_t cnt = 0;
    if (dig) {
#pragma unroll
        for (int w2 = 0; w2 < RS_WARPS; w2++) cnt += whist[w2][tid];
    }
    const uint32_t real = cnt - (((int)tid == RADIX - 1) ? (RS_TILE - nvalid) : 0u);  // padding keys are all-ones
    volatile unsigned long long *lb = lookback + (size_t)tile * RADIX + (tid & (RADIX - 1));
    if (dig) *lb = (tile == 0 ? LB_INCL : LB_LOCAL) | real;

    // block exclusive scan of cnt -> base of digit `tid` inside the tile
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31 && dig) wsum[warp] = inc;
    __syncthreads();
    uint32_t wp = 0;
#pragma unroll
    for (int w2 = 0; w2 < RADIX / 32; w2++) if (w2 < (int)warp) wp += wsum[w2];
    const uint32_t tb = wp + inc - cnt;
    // per-warp scatter base = tile base of the digit + keys of lower warps
    if (dig) {
        uint32_t run = tb;
#pragma unroll
        for (int w2 = 0; w2 < RS_WARPS; w2++) {
            const uint32_t c = whist[w2][tid];
            whist[w2][tid] = run;
            run += c;
        }
    }

    __syncthreads();

    // scatter into shared memory in tile-sorted order (needs only tile-local bases) ...
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t d = (uint32_t)(key[i] >> shift) & (uint32_t)(RADIX - 1);
        const uint32_t pos = wh[d] + rank[i];
        skeys[pos] = key[i];
        rank[i] = (uint16_t)pos;
    }
    if (HAS_VAL) {
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) svals[rank[i]] = val[i];
    }

    // ... and only then the decoupled look-back for digit `tid`: the later it runs, the more
    // predecessors already hold INCLUSIVE prefixes. Four predecessor entries are fetched per
    // step so that the walk is not one dependent L2 round trip per tile.
    unsigned long long excl = 0;
    if (tile > 0 && dig) {
        int64_t t = (int64_t)tile - 1;
        bool done = false;
        while (!done) {
            unsigned long long v[RS_LB_BATCH];
#pragma unroll
            for (int j = 0; j < RS_LB_BATCH; j++) {
                const int64_t tj = t - j;
                v[j] = tj >= 0 ? *(volatile unsigned long long *)(lookback + (size_t)tj * RADIX + tid) : LB_INCL;
            }
#pragma unroll
            for (int j = 0; j < RS_LB_BATCH; j++) {
                if (done) break;
                if ((v[j] >> 62) == 0) break;          // not published yet: re-read from here
                excl += v[j] & LB_MASK;
                t--;
                if ((v[j] >> 62) == 2) done = true;
            }
        }
        *lb = LB_INCL | (excl + real);
    }
    if (dig) goff[tid] = gbase[tid] + excl - tb;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t p = i * RS_THREADS + tid;
        if (p < nvalid) {
            const KeyT kk = skeys[p];
            const uint32_t d = (uint32_t)(kk >> shift) & (uint32_t)(RADIX - 1);
            const unsigned long long dst = goff[d] + p;
            kout[dst] = kk;
            if (HAS_VAL) vout[dst] = svals[p];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Exclusive scan u32 counts -> u64 offsets (offs[n] = total) in two launches over chunks of SCAN_CHUNK counts:
// k_scan_sums adds up every chunk, k_scan_chunks scans each chunk from the sum of the chunks before it.
#define SCAN_THREADS 1024
#define SCAN_PER 8
#define SCAN_CHUNK (SCAN_THREADS * SCAN_PER)

// block-wide sum of one value per thread (SCAN_THREADS threads); every thread gets it
__device__ __forceinline__ unsigned long long scan_block_sum(unsigned long long v, unsigned long long *ws) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) ws[warp] = v;
    __syncthreads();
    unsigned long long t = ws[lane];
#pragma unroll
    for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_sums(const uint32_t *__restrict__ counts, uint64_t n, unsigned long long *__restrict__ sums) {
    __shared__ unsigned long long ws[32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_CHUNK + threadIdx.x;
    unsigned long long v = 0;
#pragma unroll
    for (int j = 0; j < SCAN_PER; j++) {
        const uint64_t i = base + (uint64_t)j * SCAN_THREADS;
        if (i < n) v += counts[i];
    }
    v = scan_block_sum(v, ws);
    if (threadIdx.x == 0) sums[blockIdx.x] = v;
}

__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_chunks(const uint32_t *__restrict__ counts, uint64_t n, const unsigned long long *__restrict__ sums,
              unsigned long long *__restrict__ offs) {
    __shared__ unsigned long long ws[32];
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long before = 0;
    for (uint32_t b = tid; b < blockIdx.x; b += SCAN_THREADS) before += sums[b];
    before = scan_block_sum(before, ws);
    uint32_t v[SCAN_PER];
    unsigned long long tsum = 0;
    const uint64_t i0 = (uint64_t)blockIdx.x * SCAN_CHUNK + (uint64_t)tid * SCAN_PER;
#pragma unroll
    for (int j = 0; j < SCAN_PER; j++) { v[j] = (i0 + j < n) ? counts[i0 + j] : 0u; tsum += v[j]; }
    unsigned long long inc = tsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = ws[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= (unsigned)o) wi += t;
        }
        ws[lane] = wi - w;  // exclusive
    }
    __syncthreads();
    unsigned long long run = before + ws[warp] + inc - tsum;
#pragma unroll
    for (int j = 0; j < SCAN_PER; j++) { if (i0 + j < n) offs[i0 + j] = run; run += v[j]; }
    if (blockIdx.x == gridDim.x - 1 && tid == SCAN_THREADS - 1) offs[n] = run;
}

// ---------------------------------------------------------------------------------------
// Run heads of a sorted key array. One warp = one chunk of RUN_CHUNK consecutive elements.
#define RUN_CHUNK 4096
#define RUN_THREADS 256

// kshift: bits to drop before comparing (16 for packed key<<16|tag records, else 0)
template <typename KeyT>
__global__ void __launch_bounds__(RUN_THREADS)
k_run_count(const KeyT *__restrict__ keys, uint64_t n, int kshift, uint32_t *__restrict__ chunk_counts) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t chunk = (uint64_t)blockIdx.x * (RUN_THREADS / 32) + (threadIdx.x >> 5);
    const uint64_t base = chunk * RUN_CHUNK;
    if (base >= n) return;
    uint32_t c = 0;
    for (int it = 0; it < RUN_CHUNK / 32; it++) {
        const uint64_t i = base + it * 32 + lane;
        bool head = false;
        if (i < n) {
            const KeyT cur = keys[i] >> kshift;
            head = ((i == 0) || cur != (keys[i - 1] >> kshift)) && cur != (KeyT(~KeyT(0)) >> kshift);  // sentinel
        }
        c += __popc(__ballot_sync(0xffffffffu, head));
    }
    if (lane == 0) chunk_counts[chunk] = c;
}

// Per-sample run-length encode: distinct keys + head positions (counts by difference).
template <typename KeyT>
__global__ void __launch_bounds__(RUN_THREADS)
k_rle_write(const KeyT *__restrict__ keys, uint64_t n, const unsigned long long *__restrict__ chunk_offs,
            KeyT *__restrict__ out_keys, unsigned long long *__restrict__ head_pos) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t chunk = (uint64_t)blockIdx.x * (RUN_THREADS / 32) + (threadIdx.x >> 5);
    const uint64_t base = chunk * RUN_CHUNK;
    if (base >= n) return;
    unsigned long long run = chunk_offs[chunk];
    for (int it = 0; it < RUN_CHUNK / 32; it++) {
        const uint64_t i = base + it * 32 + lane;
        bool head = false;
        KeyT kk = 0;
        if (i < n) { kk = keys[i]; head = (i == 0) || kk != keys[i - 1]; }
        const unsigned ball = __ballot_sync(0xffffffffu, head);
        if (head) {
            const unsigned long long r = run + __popc(ball & lanemask_lt());
            out_keys[r] = kk;
            head_pos[r] = i;
        }
        run += __popc(ball);
    }
}

// counts[r] = head_pos[r+1] - head_pos[r]; keep flag = count >= cutoff; per-chunk kept counts
__global__ void k_rle_counts(const unsigned long long *__restrict__ head_pos, uint64_t nu, uint64_t n,
                             uint32_t cutoff, uint32_t *__restrict__ counts,
                             uint32_t *__restrict__ chunk_counts) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t chunk = (uint64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    const uint64_t base = chunk * RUN_CHUNK;
    if (base >= nu) return;
    uint32_t c = 0;
    for (int it = 0; it < RUN_CHUNK / 32; it++) {
        const uint64_t r = base + it * 32 + lane;
        bool keep = false;
        if (r < nu) {
            const unsigned long long e = (r + 1 < nu) ? head_pos[r + 1] : n;
            const uint32_t cnt = (uint32_t)(e - head_pos[r]);
            counts[r] = cnt;
            keep = cnt >= cutoff;
        }
        c += __popc(__ballot_sync(0xffffffffu, keep));
    }
    if (lane == 0) chunk_counts[chunk] = c;
}

// compact (key, count) pairs with count >= cutoff, order preserved
template <typename KeyT>
__global__ void k_rle_filter(const KeyT *__restrict__ keys, const uint32_t *__restrict__ counts, uint64_t nu,
                             uint32_t cutoff, const unsigned long long *__restrict__ chunk_offs,
                             KeyT *__restrict__ out_keys, uint32_t *__restrict__ out_counts) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t chunk = (uint64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    const uint64_t base = chunk * RUN_CHUNK;
    if (base >= nu) return;
    unsigned long long run = chunk_offs[chunk];
    for (int it = 0; it < RUN_CHUNK / 32; it++) {
        const uint64_t r = base + it * 32 + lane;
        bool keep = false;
        uint32_t cnt = 0;
        if (r < nu) { cnt = counts[r]; keep = cnt >= cutoff; }
        const unsigned ball = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const unsigned long long o = run + __popc(ball & lanemask_lt());
            out_keys[o] = keys[r];
            out_counts[o] = cnt;
        }
        run += __popc(ball);
    }
}
