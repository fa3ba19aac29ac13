// ps_count.cuh — occurrence counts of K query k-mers in every sample of a block (ps_count_matrix, ps_lookup).
//
// Replaces `gmer_counter -db` per sample (prediction.py:72-100) and the per-sample lookups of `-rc`
// (modeling.py:693-695): one pass over the decoded 2-bit streams of the selected samples gives an N x K matrix.
//
//   k_count_filter   sets 2 bits per unique query in one 32-bit word of a 2^20-bit blocked Bloom filter (global).
//   k_count_matrix   persistent blocks, one per SM: the filter is copied into 128 KB of shared memory once per
//                    block, then warps take 512-position units of the selected samples' streams (grid stride).
//                    Lane l owns 16 consecutive positions, computes their canonical k-mers from its stream words
//                    with funnel shifts and a reverse complement taken once (as k_scatter1), and probes the
//                    filter: a miss costs one shared-memory load. A hit looks the key up in the sorted unique
//                    queries (a radix index on the top 16 key bits, then a binary search, both in L2) and
//                    adds 1 to counts[row * Ku + q].
//   k_count_expand   unique-query counts -> the caller's query order (duplicates, unsorted queries).
#pragma once
#include "ps_common.cuh"
#include "ps_extract.cuh"

#define CNT_THREADS 1024
#define CNT_FILTER_LOG2_WORDS 15
#define CNT_FILTER_WORDS (1u << CNT_FILTER_LOG2_WORDS)      // 32768 words = 128 KB = 2^20 bits
#define CNT_INDEX_BITS 16                                   // radix index over the top key bits
#define CNT_UNIT 512                                        // positions of one warp unit (8 per 4096-block)

// filter word and bit pair of one canonical k-mer: Fibonacci hash, word from the top 15 bits, bits from the low 10
__device__ __forceinline__ uint32_t cnt_hash(uint64_t key) { return (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 32); }
__device__ __forceinline__ uint32_t cnt_word(uint32_t h) { return h >> (32 - CNT_FILTER_LOG2_WORDS); }
__device__ __forceinline__ uint32_t cnt_bits(uint32_t h) { return (1u << (h & 31u)) | (1u << ((h >> 5) & 31u)); }

__global__ void k_count_filter(const uint64_t *__restrict__ q, uint64_t n, uint32_t *__restrict__ filter) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t h = cnt_hash(q[i]);
        atomicOr(filter + cnt_word(h), cnt_bits(h));
    }
}

struct CntArgs {
    const uint32_t *seq, *bad;          // the stream pool
    const uint64_t *blk_first;          // per row: first pool block (4096 positions) of the sample
    const uint32_t *blk_prefix;         // per row: stream blocks of the rows before it; [nrows] = all of them
    int nrows;
    int k;
    const uint32_t *filter;             // CNT_FILTER_WORDS
    const uint64_t *queries;            // Ku ascending unique canonical k-mers
    const uint32_t *qidx;               // (1 << ibits) + 1: first query whose key >> ishift is >= i
    int ishift;
    uint64_t Ku;
    uint32_t *counts;                   // nrows x Ku
};

__device__ __forceinline__ void cnt_probe(const CntArgs &a, const uint32_t *s_filter, uint32_t *crow, uint64_t key) {
    const uint32_t h = cnt_hash(key), bits = cnt_bits(h);
    if ((s_filter[cnt_word(h)] & bits) != bits) return;
    const uint32_t top = (uint32_t)(key >> a.ishift);
    uint32_t lo = __ldg(a.qidx + top);
    const uint32_t end = __ldg(a.qidx + top + 1);
    uint32_t hi = end;
    while (lo < hi) {
        const uint32_t m = (lo + hi) >> 1;
        if (__ldg(a.queries + m) < key) lo = m + 1; else hi = m;
    }
    if (lo < end && __ldg(a.queries + lo) == key) atomicAdd(crow + lo, 1u);
}

template <typename KeyT>
__global__ void __launch_bounds__(CNT_THREADS, 1) k_count_matrix(CntArgs a) {
    extern __shared__ __align__(16) uint32_t s_filter[];
    for (uint32_t i = threadIdx.x; i < CNT_FILTER_WORDS / 4; i += CNT_THREADS)
        reinterpret_cast<uint4 *>(s_filter)[i] = __ldg(reinterpret_cast<const uint4 *>(a.filter) + i);
    __syncthreads();
    const unsigned lane = threadIdx.x & 31;
    const int k = a.k;
    const uint64_t kmask = (1ull << k) - 1ull;
    const uint64_t units = (uint64_t)__ldg(a.blk_prefix + a.nrows) * (EXT_BLOCK_POS / CNT_UNIT);
    const uint64_t nwarps = (uint64_t)gridDim.x * (CNT_THREADS / 32);
    int row = 0;
    for (uint64_t u = blockIdx.x * (uint64_t)(CNT_THREADS / 32) + (threadIdx.x >> 5); u < units; u += nwarps) {
        const uint32_t b = (uint32_t)(u / (EXT_BLOCK_POS / CNT_UNIT));
        // the row holding stream block b: last r with blk_prefix[r] <= b (units only move forward)
        int hi = a.nrows;
        while (hi - row > 1) {
            const int m = (row + hi) >> 1;
            if (__ldg(a.blk_prefix + m) <= b) row = m; else hi = m;
        }
        const uint64_t base = (__ldg(a.blk_first + row) + (b - __ldg(a.blk_prefix + row))) * EXT_BLOCK_POS +
                              (u % (EXT_BLOCK_POS / CNT_UNIT)) * CNT_UNIT + 16 * lane;
        uint32_t *crow = a.counts + (uint64_t)row * a.Ku;
        // lane's positions base .. base + 15; windows reach at most 31 positions further (3 stream words, 48 mask bits)
        const uint32_t *sp = a.seq + (base >> 4);
        const uint32_t *bp = a.bad + (base >> 5);
        const uint64_t badwin = ((uint64_t)__ldg(bp + 1) << 32 | __ldg(bp)) >> (base & 31);
        const uint32_t w0 = __ldg(sp), w1 = __ldg(sp + 1);
        if (sizeof(KeyT) == 4) {
            // as k_scatter1: the reverse complement of the 32 bases once, pre-shifted so that the window at `it`
            // is one funnel shift by a compile-time amount
            const int dn = 32 - 2 * k;
            const uint64_t rcw = (((uint64_t)rev2_32(~w1) << 32) | (uint64_t)rev2_32(~w0)) << (34 - 2 * k);
            const uint32_t rc_hi = (uint32_t)(rcw >> 32), rc_lo = (uint32_t)rcw;
#pragma unroll
            for (int it = 0; it < 16; it++) {
                if ((badwin >> it) & kmask) continue;
                const uint32_t fw = __funnelshift_l(w1, w0, 2 * it) >> dn;
                const uint32_t rc = __funnelshift_l(rc_lo, rc_hi, 30 - 2 * it) >> dn;
                cnt_probe(a, s_filter, crow, fw < rc ? fw : rc);
            }
        } else {
            // 48 bases in three words; their reverse complement r2:r1:r0 (base 47 - j at index j) is pre-shifted
            // left by 2 (33 - k) bits, so that the window at `it` starts 15 - it bases into it
            const uint32_t w2 = __ldg(sp + 2);
            const uint32_t r2 = rev2_32(~w2), r1 = rev2_32(~w1), r0 = rev2_32(~w0);
            const uint32_t p = 2 * (33 - k);
            const uint32_t A = __funnelshift_lc(r1, r2, p), B = __funnelshift_lc(r0, r1, p), C = __funnelshift_lc(0u, r0, p);
            const int dn = 64 - 2 * k;
#pragma unroll
            for (int it = 0; it < 16; it++) {
                if ((badwin >> it) & kmask) continue;
                const uint64_t fw = (((uint64_t)__funnelshift_l(w1, w0, 2 * it) << 32) | __funnelshift_l(w2, w1, 2 * it)) >> dn;
                const uint64_t rc = (((uint64_t)__funnelshift_l(B, A, 30 - 2 * it) << 32) | __funnelshift_l(C, B, 30 - 2 * it)) >> dn;
                cnt_probe(a, s_filter, crow, fw < rc ? fw : rc);
            }
        }
    }
}

// out[r * K + j] = cnt[r * Ku + inv[j]]
__global__ void k_count_expand(const uint32_t *__restrict__ cnt, uint64_t Ku, const uint32_t *__restrict__ inv,
                               uint64_t K, uint64_t n, uint32_t *__restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = cnt[(i / K) * Ku + inv[i % K]];
}
