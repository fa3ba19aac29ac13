// ps_extract.cuh — canonical k-mer extraction from the 2-bit packed stream pool.
//
// Replaces the k-mer enumeration half of `glistmaker` (modeling.py:303-315): every stream
// position q whose window [q, q+k) holds no invalid position yields
// canonical = min(word, revcomp(word)), 2 bits/base, first base most significant.
// k <= 16 packs into u32 keys, k <= 32 into u64 keys.
//
// One block = 4096 consecutive positions (never straddles samples: streams are padded to
// 4096). Warp w walks 512 positions in 16 coalesced steps; valid & in-range k-mers are
// compacted in stream order (ballot + popc), so the output order is deterministic and a
// stable sort keeps every sample's instances of one k-mer adjacent.
#pragma once
#include "ps_common.cuh"

#define EXT_THREADS 256
#define EXT_ITERS 16
#define EXT_BLOCK_POS (EXT_THREADS * EXT_ITERS)  // 4096 == POS_ALIGN

template <typename KeyT> struct KeyTraits;
template <> struct KeyTraits<uint32_t> { static constexpr int BITS = 32; };
template <> struct KeyTraits<uint64_t> { static constexpr int BITS = 64; };

__device__ __forceinline__ uint32_t rev2_32(uint32_t x) {
    x = __brev(x);
    return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}
__device__ __forceinline__ uint64_t rev2_64(uint64_t x) {
    x = __brevll(x);
    return ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
}

// Canonical k-mer starting at pool position q; returns false if the window is invalid.
template <typename KeyT>
__device__ __forceinline__ bool kmer_at(const uint32_t *__restrict__ seq,
                                        const uint32_t *__restrict__ bad, uint64_t q, int k,
                                        KeyT &out) {
    const uint64_t mw = q >> 5;
    const uint32_t m0 = __ldg(bad + mw), m1 = __ldg(bad + mw + 1);
    const uint32_t win = __funnelshift_r(m0, m1, (uint32_t)(q & 31));
    const uint32_t kmask = k == 32 ? 0xFFFFFFFFu : ((1u << k) - 1u);
    if (win & kmask) return false;
    const uint64_t sw = q >> 4;
    const uint32_t sh = 2u * (uint32_t)(q & 15);
    const uint32_t w0 = __ldg(seq + sw), w1 = __ldg(seq + sw + 1);
    if (sizeof(KeyT) == 4) {
        const uint32_t f32 = __funnelshift_l(w1, w0, sh);
        const uint32_t fw = f32 >> (32 - 2 * k);
        const uint32_t rc = rev2_32(~fw) >> (32 - 2 * k);
        out = (KeyT)(fw < rc ? fw : rc);
    } else {
        const uint32_t w2 = __ldg(seq + sw + 2);
        const uint64_t f64 = ((uint64_t)__funnelshift_l(w1, w0, sh) << 32) | __funnelshift_l(w2, w1, sh);
        const uint64_t fw = f64 >> (64 - 2 * k);
        const uint64_t rc = rev2_64(~fw) >> (64 - 2 * k);
        out = (KeyT)(fw < rc ? fw : rc);
    }
    return true;
}

// COUNT pass: per-block number of valid in-range k-mers.
// WRITE pass: compacted keys at blk_offs[block]. TAGS 0: keys only; 1: keys + u16 sample tags
// (two arrays); 2: packed 64-bit records (key << 16 | tag) written through keys_out.
template <typename KeyT, bool WRITE, int TAGS>
__global__ void __launch_bounds__(EXT_THREADS)
k_extract(const uint32_t *__restrict__ seq, const uint32_t *__restrict__ bad, uint64_t pos_begin,
          int k, uint64_t lo, uint64_t hi, int range_all, const uint16_t *__restrict__ blk_sample,
          uint32_t *__restrict__ blk_counts, const uint64_t *__restrict__ blk_offs,
          KeyT *__restrict__ keys_out, uint16_t *__restrict__ tags_out) {
    __shared__ uint32_t wsum[EXT_THREADS / 32];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t base = pos_begin + (uint64_t)blockIdx.x * EXT_BLOCK_POS + warp * (32 * EXT_ITERS);
    KeyT keys[EXT_ITERS];
    uint32_t validbits = 0, wcount = 0;
    uint16_t off[EXT_ITERS];
#pragma unroll
    for (int it = 0; it < EXT_ITERS; it++) {
        KeyT key = 0;
        bool ok = kmer_at<KeyT>(seq, bad, base + it * 32 + lane, k, key);
        if (ok && !range_all) ok = (uint64_t)key >= lo && (uint64_t)key < hi;
        const unsigned ball = __ballot_sync(0xffffffffu, ok);
        if (WRITE) {
            keys[it] = key;
            off[it] = (uint16_t)(wcount + __popc(ball & lanemask_lt()));
            validbits |= (ok ? 1u : 0u) << it;
        }
        wcount += __popc(ball);
    }
    if (lane == 0) wsum[warp] = wcount;
    __syncthreads();
    if (!WRITE) {
        if (threadIdx.x == 0) {
            uint32_t s = 0;
#pragma unroll
            for (int w2 = 0; w2 < EXT_THREADS / 32; w2++) s += wsum[w2];
            blk_counts[blockIdx.x] = s;
        }
        return;
    }
    uint64_t o = blk_offs[blockIdx.x];
    for (unsigned w2 = 0; w2 < warp; w2++) o += wsum[w2];
    const uint16_t tag = TAGS ? blk_sample[(pos_begin >> 12) + blockIdx.x] : 0;
#pragma unroll
    for (int it = 0; it < EXT_ITERS; it++) {
        if ((validbits >> it) & 1u) {
            if (TAGS == 2) {
                reinterpret_cast<uint64_t *>(keys_out)[o + off[it]] = ((uint64_t)keys[it] << 16) | tag;
            } else {
                keys_out[o + off[it]] = keys[it];
                if (TAGS == 1) tags_out[o + off[it]] = tag;
            }
        }
    }
}

#define PART_MAX 8   // GPUs of one routed job (ps_paged.cuh)

// Gather per-sample counted lists (list mode) into the instance arrays, range-filtered, in
// list order. One block handles 4096 list entries of one sample (lists padded likewise).
template <typename KeyT, bool WRITE, int TAGS>
__global__ void __launch_bounds__(EXT_THREADS)
k_list_gather(const KeyT *__restrict__ list_keys, uint64_t ent_begin, uint64_t lo, uint64_t hi,
              int range_all, const uint16_t *__restrict__ blk_sample,
              const uint32_t *__restrict__ blk_valid, uint32_t *__restrict__ blk_counts,
              const uint64_t *__restrict__ blk_offs, KeyT *__restrict__ keys_out,
              uint16_t *__restrict__ tags_out) {
    __shared__ uint32_t wsum[EXT_THREADS / 32];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t base = ent_begin + (uint64_t)blockIdx.x * EXT_BLOCK_POS + warp * (32 * EXT_ITERS);
    const uint32_t nvalid = blk_valid[blockIdx.x];  // valid entries in this block
    KeyT keys[EXT_ITERS];
    uint32_t validbits = 0, wcount = 0;
    uint16_t off[EXT_ITERS];
#pragma unroll
    for (int it = 0; it < EXT_ITERS; it++) {
        const uint32_t li = warp * (32 * EXT_ITERS) + it * 32 + lane;
        KeyT key = 0;
        bool ok = li < nvalid;
        if (ok) {
            key = list_keys[base + it * 32 + lane];
            if (!range_all) ok = (uint64_t)key >= lo && (uint64_t)key < hi;
        }
        const unsigned ball = __ballot_sync(0xffffffffu, ok);
        if (WRITE) {
            keys[it] = key;
            off[it] = (uint16_t)(wcount + __popc(ball & lanemask_lt()));
            validbits |= (ok ? 1u : 0u) << it;
        }
        wcount += __popc(ball);
    }
    if (lane == 0) wsum[warp] = wcount;
    __syncthreads();
    if (!WRITE) {
        if (threadIdx.x == 0) {
            uint32_t s = 0;
            for (int w2 = 0; w2 < EXT_THREADS / 32; w2++) s += wsum[w2];
            blk_counts[blockIdx.x] = s;
        }
        return;
    }
    uint64_t o = blk_offs[blockIdx.x];
    for (unsigned w2 = 0; w2 < warp; w2++) o += wsum[w2];
    const uint16_t tag = blk_sample[blockIdx.x];
#pragma unroll
    for (int it = 0; it < EXT_ITERS; it++) {
        if ((validbits >> it) & 1u) {
            if (TAGS == 2) {
                reinterpret_cast<uint64_t *>(keys_out)[o + off[it]] = ((uint64_t)keys[it] << 16) | tag;
            } else {
                keys_out[o + off[it]] = keys[it];
                tags_out[o + off[it]] = tag;
            }
        }
    }
}
