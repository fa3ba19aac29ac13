// ps_mash.cuh — `-w` sample weights on the device: MinHash sketches of the decoded streams, the (shared, denom)
// counts of every sketch pair, and neighbour joining in FP64. The O(N) GSC tree arithmetic stays on the host
// (phenotypeseeker_b200/weights.py), which also restates every step here for the tests.
//
// Replaces: `mash sketch -r` (modeling.py:386-390), `mash paste` + `mash dist` (:404-412) and Biopython's
// DistanceTreeConstructor.nj (:446-452).
#pragma once
#include "ps_common.cuh"
#include "ps_extract.cuh"
#include "ps_mash_bits.h"

#define MASH_THREADS 256
#define MASH_ROUND (MASH_THREADS * 16)    // positions hashed by one block between two threshold checks

// u64 slots of the shared bottom list + candidate buffer: a power of two with room for s, one round of candidates and
// 1024 more, so that a full bottom list is reduced again only after another 1024+ candidates (s = 1000: 8192, 64 KB)
static inline int mash_cap(int s) {
    int cap = 8192;
    while (cap < s + MASH_ROUND + 1024) cap <<= 1;
    return cap;
}
static inline size_t mash_smem(int s) { return (size_t)(mash_cap(s) + s) * 8; }

// ---- block-wide helpers over a shared array of u64 ----------------------------------------------------------------
// In-place ascending bitonic sort of a[0..n2), n2 a power of two.
__device__ __forceinline__ void mash_bitonic(uint64_t *a, int n2) {
    for (int size = 2; size <= n2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < (n2 >> 1); t += blockDim.x) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool up = (lo & size) == 0;
                const uint64_t x = a[lo], y = a[hi];
                if ((x > y) == up) { a[lo] = y; a[hi] = x; }
            }
            __syncthreads();
        }
    }
}

// a[0..n) holds the current bottom list followed by candidates, in any order. Leaves in a[0..*nb) the ascending
// bottom-s distinct values of a[0..n) and returns that count. `out` is scratch of s entries; `wtot` of 32 words.
// a must have room for the next power of two >= n. Call with the whole block; returns the same value everywhere.
__device__ int mash_reduce(uint64_t *a, int n, int s, uint64_t *out, uint32_t *wtot) {
    int n2 = 64;
    while (n2 < n) n2 <<= 1;
    for (int i = n + threadIdx.x; i < n2; i += blockDim.x) a[i] = ~0ull;
    __syncthreads();
    mash_bitonic(a, n2);
    // rank of every first occurrence among the first n values: per-thread runs of `per` consecutive values
    const int per = (n + blockDim.x - 1) / blockDim.x;
    const int b0 = threadIdx.x * per, b1 = min(n, b0 + per);
    uint32_t mine = 0;
    for (int i = b0; i < b1; i++) mine += (i == 0 || a[i] != a[i - 1]);
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = mine;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += v;
    }
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    uint32_t base = inc - mine, total = 0;
    for (unsigned w = 0; w < blockDim.x / 32; w++) {
        if (w < warp) base += wtot[w];
        total += wtot[w];
    }
    for (int i = b0; i < b1 && base < (uint32_t)s; i++)
        if (i == 0 || a[i] != a[i - 1]) out[base++] = a[i];
    __syncthreads();
    const int keep = min((int)total, s);
    for (int i = threadIdx.x; i < keep; i += blockDim.x) a[i] = out[i];
    __syncthreads();
    return keep;
}

// ---- k_mash_sketch: grid (chunk, sample) ----------------------------------------------------------------------------
// Block (c, i) hashes every valid k-window that starts in chunk c of sample i's stream (chunk_pos positions, a multiple
// of MASH_ROUND) and writes the ascending bottom-s distinct hashes to out[(i * n_chunks + c) * s ..], count to
// out_n[i * n_chunks + c]. Shared memory: cap u64 (bottom list + candidate buffer, cap a power of two >= s + 2 *
// MASH_ROUND) + s u64 scratch. Thread t owns positions 16 t .. 16 t + 15 of a round: it loads the three stream words
// and two break words that cover its 16 windows once and funnel-shifts every window out of them.
__global__ void __launch_bounds__(MASH_THREADS)
k_mash_sketch(const uint32_t *__restrict__ seq, const uint32_t *__restrict__ bad, const uint64_t *__restrict__ s_off,
              const uint64_t *__restrict__ s_npos, int n_chunks, uint64_t chunk_pos, int k, int s, int cap, uint32_t seed,
              uint64_t *__restrict__ out, uint32_t *__restrict__ out_n) {
    extern __shared__ uint64_t sm_mash[];
    uint64_t *a = sm_mash, *scratch = sm_mash + cap;
    __shared__ uint32_t wtot[32];
    __shared__ int cnt;
    const int i = blockIdx.y, c = blockIdx.x;
    const uint64_t npos = s_npos[i];
    const uint64_t p0 = (uint64_t)c * chunk_pos;
    uint32_t *dst_n = out_n + (size_t)i * n_chunks + c;
    if (p0 >= npos) {
        if (threadIdx.x == 0) *dst_n = 0;
        return;
    }
    const uint64_t p1 = min(npos, p0 + chunk_pos);
    const uint64_t base = s_off[i];
    const uint32_t kmask = k == 32 ? 0xFFFFFFFFu : ((1u << k) - 1u);
    int nb = 0;                    // values in the bottom list a[0..nb)
    bool full = false;
    uint64_t tau = ~0ull;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (uint64_t r0 = p0; r0 < p1; r0 += MASH_ROUND) {
        const uint64_t q = base + r0 + 16u * threadIdx.x;        // first position of this thread, multiple of 16
        const uint64_t sw = q >> 4, mw = q >> 5;
        const uint32_t w0 = __ldg(seq + sw), w1 = __ldg(seq + sw + 1), w2 = __ldg(seq + sw + 2);
        const uint64_t bw = ((uint64_t)__ldg(bad + mw + 1) << 32 | __ldg(bad + mw)) >> (q & 31);
#pragma unroll 4
        for (int j = 0; j < 16; j++) {
            if ((uint32_t)(bw >> j) & kmask) continue;
            const uint32_t sh = 2u * j;
            const uint64_t f64 = ((uint64_t)__funnelshift_l(w1, w0, sh) << 32) | __funnelshift_l(w2, w1, sh);
            const uint64_t h = psm_hash_kmer(psm_canonical(f64 >> (64 - 2 * k), k), k, seed);
            if (!full || h < tau) a[nb + atomicAdd(&cnt, 1)] = h;
        }
        __syncthreads();
        const int added = cnt, n = nb + added;
        __syncthreads();                                          // everyone has read cnt before it changes again
        if (n > cap - MASH_ROUND || (r0 + MASH_ROUND >= p1 && added > 0)) {   // no room for another round, or the end
            nb = mash_reduce(a, n, s, scratch, wtot);
            full = nb == s;
            tau = full ? a[s - 1] : ~0ull;
            if (threadIdx.x == 0) cnt = 0;
            __syncthreads();
        }
    }
    uint64_t *dst = out + ((size_t)i * n_chunks + c) * s;
    for (int t = threadIdx.x; t < nb; t += blockDim.x) dst[t] = a[t];
    if (threadIdx.x == 0) *dst_n = nb;
}

// ---- k_mash_merge: one block per sample ----------------------------------------------------------------------------
// The bottom-s distinct of a union lies in the union of its parts' bottom-s distinct, so merging the chunk lists is
// exact. Chunk lists are appended behind the running bottom list while they fit, then reduced.
__global__ void __launch_bounds__(MASH_THREADS)
k_mash_merge(const uint64_t *__restrict__ parts, const uint32_t *__restrict__ parts_n, int n_chunks, int s, int cap,
             uint64_t *__restrict__ hashes, uint32_t *__restrict__ n_hashes) {
    extern __shared__ uint64_t sm_mash[];
    uint64_t *a = sm_mash, *scratch = sm_mash + cap;
    __shared__ uint32_t wtot[32];
    const int i = blockIdx.x;
    int n = 0;
    for (int c = 0; c < n_chunks; c++) {
        const uint32_t m = parts_n[(size_t)i * n_chunks + c];
        if (n + (int)m > cap) {
            n = mash_reduce(a, n, s, scratch, wtot);
        }
        const uint64_t *src = parts + ((size_t)i * n_chunks + c) * s;
        for (uint32_t t = threadIdx.x; t < m; t += blockDim.x) a[n + t] = src[t];
        n += m;
        __syncthreads();
    }
    if (n) n = mash_reduce(a, n, s, scratch, wtot);
    for (int t = threadIdx.x; t < n; t += blockDim.x) hashes[(size_t)i * s + t] = a[t];
    if (threadIdx.x == 0) n_hashes[i] = n;
}

// ---- k_mash_pairs: grid (tile of 256 j, i) --------------------------------------------------------------------------
// Sketch i is staged in shared memory; thread j >= i walks the merge of sketch i and sketch j exactly as `mash dist`
// does (psm_shared_denom) and writes the result to both (i, j) and (j, i).
__global__ void __launch_bounds__(256)
k_mash_pairs(const uint64_t *__restrict__ hashes, const uint32_t *__restrict__ n_hashes, int n, int s,
             uint32_t *__restrict__ sd) {
    extern __shared__ uint64_t sm_mash[];
    const int i = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if ((int)(blockIdx.x * blockDim.x + blockDim.x) <= i) return;     // whole tile below the diagonal
    const uint32_t na = n_hashes[i];
    for (uint32_t t = threadIdx.x; t < na; t += blockDim.x) sm_mash[t] = hashes[(size_t)i * s + t];
    __syncthreads();
    if (j < i || j >= n) return;
    const uint32_t v = psm_shared_denom(sm_mash, na, hashes + (size_t)j * s, n_hashes[j], (uint32_t)s);
    sd[(size_t)i * n + j] = v;
    sd[(size_t)j * n + i] = v;
}

// ---- neighbour joining ----------------------------------------------------------------------------------------------
// D: FP64, row stride ld, symmetric in physical slots. act[p] = slot of list position p (increasing in p). One step
// restates one iteration of weights.nj_joins with m active positions, in three launches:
//   k_nj_rowsum:  nd[p] = (sum over x of D[act[p]][act[x]] in list order, summed as Python's sum() does:
//                 psm_sum_*, compensated) / (m - 2), one thread per p;
//                 D is symmetric, so the thread reads column act[p] of rows act[x], coalesced across p.
//   k_nj_argmin:  per block, the first (i, j), j < i, in (i, j) order with the smallest (D[i][j] - nd[i]) - nd[j].
//   k_nj_update:  every block reduces the block minima to (mi, mj); then D row and column mj = the inner node,
//                 the branch lengths, and act without position mi (into act_next). mi > mj, except for a
//                 minimum first reached at pair (1, 0), which joins as (0, 1); either way the slots stay increasing.
__global__ void __launch_bounds__(128)
k_nj_rowsum(const double *__restrict__ D, size_t ld, const int *__restrict__ act, int m, double *__restrict__ nd) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    const double *col = D + act[p];
    PsmSum sum;
    psm_sum_first(sum, col[(size_t)act[0] * ld]);
    int x = 1;
    for (; x + 8 <= m; x += 8) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = col[(size_t)act[x + u] * ld];
#pragma unroll
        for (int u = 0; u < 8; u++) psm_sum_add(sum, v[u]);
    }
    for (; x < m; x++) psm_sum_add(sum, col[(size_t)act[x] * ld]);
    nd[p] = psm_sum_end(sum) / (double)(m - 2);
}

struct NjBest {
    double t;
    uint64_t key;    // i << 32 | j
};

__device__ __forceinline__ bool nj_better(double t, uint64_t key, double bt, uint64_t bkey) {
    return t < bt || (t == bt && key < bkey);
}

__device__ __forceinline__ void nj_warp_min(double &t, uint64_t &key) {
    for (int o = 16; o > 0; o >>= 1) {
        const double t2 = __shfl_down_sync(0xffffffffu, t, o);
        const uint64_t k2 = __shfl_down_sync(0xffffffffu, key, o);
        if (nj_better(t2, k2, t, key)) { t = t2; key = k2; }
    }
}

// one warp per row i (1 <= i < m), lanes over j < i; block minimum -> part[blockIdx.x]
__global__ void __launch_bounds__(256)
k_nj_argmin(const double *__restrict__ D, size_t ld, const int *__restrict__ act, int m, const double *__restrict__ nd,
            NjBest *__restrict__ part) {
    __shared__ double st[8];
    __shared__ uint64_t sk[8];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = gridDim.x * (blockDim.x >> 5);
    double bt = __longlong_as_double(0x7FF0000000000000ll);   // +inf
    uint64_t bkey = ~0ull;
    for (int i = 1 + blockIdx.x * (blockDim.x >> 5) + warp; i < m; i += nwarps) {
        const double *row = D + (size_t)act[i] * ld;
        const double ndi = nd[i];
        for (int j = lane; j < i; j += 32) {
            const double t = (row[act[j]] - ndi) - nd[j];
            const uint64_t key = (uint64_t)i << 32 | (uint32_t)j;
            if (nj_better(t, key, bt, bkey)) { bt = t; bkey = key; }
        }
    }
    nj_warp_min(bt, bkey);
    if (lane == 0) { st[warp] = bt; sk[warp] = bkey; }
    __syncthreads();
    if (warp == 0) {
        bt = lane < (blockDim.x >> 5) ? st[lane] : __longlong_as_double(0x7FF0000000000000ll);
        bkey = lane < (blockDim.x >> 5) ? sk[lane] : ~0ull;
        nj_warp_min(bt, bkey);
        if (lane == 0) part[blockIdx.x] = NjBest{bt, bkey};
    }
}

__global__ void __launch_bounds__(256)
k_nj_update(double *__restrict__ D, size_t ld, const int *__restrict__ act, int *__restrict__ act_next, int m,
            const double *__restrict__ nd, const NjBest *__restrict__ part, int n_part, int step,
            int32_t *__restrict__ join, double *__restrict__ branch) {
    __shared__ double st[8];
    __shared__ uint64_t sk[8];
    __shared__ uint64_t best;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double bt = __longlong_as_double(0x7FF0000000000000ll);
    uint64_t bkey = ~0ull;
    for (int b = threadIdx.x; b < n_part; b += blockDim.x)
        if (nj_better(part[b].t, part[b].key, bt, bkey)) { bt = part[b].t; bkey = part[b].key; }
    nj_warp_min(bt, bkey);
    if (lane == 0) { st[warp] = bt; sk[warp] = bkey; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (unsigned w = 1; w < (blockDim.x >> 5); w++)
            if (nj_better(st[w], sk[w], st[0], sk[0])) { st[0] = st[w]; sk[0] = sk[w]; }
        best = sk[0];
    }
    __syncthreads();
    // the host loop starts from (mi, mj) = (0, 1) with the value of pair (1, 0) and moves on a strictly smaller value
    // only, so a minimum first reached at (1, 0) joins with mi = 0, mj = 1
    int mi = (int)(best >> 32), mj = (int)(uint32_t)best;
    if (mi == 1 && mj == 0) { mi = 0; mj = 1; }
    const size_t si = act[mi], sj = act[mj];
    const double dij = D[si * ld + sj];
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x == 0) {
        const double c1 = ((dij + nd[mi]) - nd[mj]) / 2.0;
        join[2 * step] = mi;
        join[2 * step + 1] = mj;
        branch[2 * step] = c1;
        branch[2 * step + 1] = dij - c1;
    }
    if (x < m) {
        if (x != mi && x != mj) {
            const size_t sx = act[x];
            const double v = ((D[si * ld + sx] + D[sj * ld + sx]) - dij) / 2.0;
            D[sj * ld + sx] = v;
            D[sx * ld + sj] = v;
        }
        if (x < m - 1) act_next[x] = act[x < mi ? x : x + 1];
    }
}

// D2[p][q] = D[act[p]][act[q]]: drops the slots of joined positions so that rows stay dense
__global__ void k_nj_compact(const double *__restrict__ D, size_t ld, const int *__restrict__ act, int m,
                             double *__restrict__ D2) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (q < m) D2[(size_t)p * m + q] = D[(size_t)act[p] * ld + act[q]];
}
