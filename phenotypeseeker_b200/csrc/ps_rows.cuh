// ps_rows.cuh — sorted (k-mer, sample) instances -> union k-mer array + k-mer-major bit matrix.
//
// Replaces `glistcompare -u` (modeling.py:351-380: the union, ascending = feature_vector.list
// order), `glistquery -l` + `split` (modeling.py:317-348: per-sample presence of every union
// k-mer) and the presence binarisation of get_kmers_tested (modeling.py:693-695).
//
// Row r of the matrix belongs to union k-mer r; sample s is bit (s & 31) of word (s >> 5);
// rows are `wp` words apart (multiple of 4 => 16-byte aligned rows for 128-bit loads).
// Duplicate instances of one (k-mer, sample) are dropped with a neighbour compare, the bits
// of one 32-instance step are merged per (row, word) with __match_any_sync +
// __reduce_or_sync, and one atomicOr per distinct (row, word) reaches memory.
#pragma once
#include "ps_common.cuh"
#include "ps_sort.cuh"
#include "ps_paged.cuh"

// PACKED: `keys` holds 64-bit records (key << 16 | tag) and `tags` is unused.
template <typename KeyT, bool PACKED>
__global__ void __launch_bounds__(RUN_THREADS)
k_row_build(const KeyT *__restrict__ keys, const uint16_t *__restrict__ tags, uint64_t n,
            const unsigned long long *__restrict__ chunk_offs, uint64_t *__restrict__ union_out,
            uint32_t *__restrict__ matrix, int wp) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t chunk = (uint64_t)blockIdx.x * (RUN_THREADS / 32) + (threadIdx.x >> 5);
    const uint64_t base = chunk * RUN_CHUNK;
    if (base >= n) return;
    unsigned long long run = chunk_offs[chunk];  // heads before this chunk
    for (int it = 0; it < RUN_CHUNK / 32; it++) {
        const uint64_t i = base + it * 32 + lane;
        const bool valid = i < n;
        KeyT kk = 0;
        uint16_t tag = 0;
        bool head = false, dup = false;
        if (valid) {
            if (PACKED) {
                const KeyT rec = keys[i];
                kk = rec >> 16;
                tag = (uint16_t)(rec & 0xFFFFu);
                if (i == 0) head = true;
                else {
                    const KeyT prev = keys[i - 1];
                    head = kk != (prev >> 16);
                    dup = rec == prev;
                }
            } else {
                kk = keys[i];
                tag = tags[i];
                if (i == 0) head = true;
                else {
                    head = kk != keys[i - 1];
                    dup = !head && tags[i - 1] == tag;
                }
            }
        }
        const unsigned ball = __ballot_sync(0xffffffffu, head);
        const uint32_t delta = __popc(ball & lanemask_le());  // heads up to and including me
        const unsigned long long row = run + delta - 1;       // valid lanes only
        if (head) union_out[row] = (uint64_t)kk;
        const bool active = valid && !dup;
        const uint32_t word = tag >> 5;
        const uint32_t id = active ? ((delta << 11) | word) : 0xFFFFFFFFu;
        const unsigned grp = __match_any_sync(0xffffffffu, id);
        const uint32_t bits = __reduce_or_sync(grp, active ? (1u << (tag & 31)) : 0u);
        if (active && (int)lane == __ffs(grp) - 1) atomicOr(matrix + row * (uint64_t)wp + word, bits);
        run += __popc(ball);
    }
}

// ---------------------------------------------------------------------------------------
// Bucketed build (2k in (16, 32]): ps_paged.cuh brings the instances of one top-16-bit prefix
// together (a bucket = all records sharing those bits, in arbitrary order, as a list of pages).
// One block owns one bucket and never sorts it: the low
// `lbits` = 2k - 16 bits of a k-mer index a presence bitmap in shared memory (<= 8 KB), whose
// prefix popcounts ARE the ranks of the distinct k-mers, i.e. their rows relative to the
// bucket's first row. k_bucket_count leaves the number of distinct k-mers per bucket and the
// bitmap itself; a scan turns the counts into first rows (and U); k_bucket_build reloads the
// bitmap, ranks it, writes the union slice and assembles the rows with shared-memory atomicOr,
// stored once. A bucket with more rows than the shared row table holds is done in row windows
// (its records re-read from L2); the largest buckets get their own launch with one block per SM
// and all of its shared memory. Union order = bucket order, then bitmap order = ascending
// k-mers = feature_vector.list order. Bucket sizes are heavy-tailed (AT-rich prefixes): blocks
// take buckets through `order`, large ones first, so that no long bucket is left for the tail.
#define BK_BITS 16
#define BK_N (1 << BK_BITS)
#define BK_THREADS 512          // k_bucket_count, k_bucket_build on ordinary buckets
#define BK_MAX_THREADS 1024     // k_bucket_build on the largest buckets (one block per SM, ~220 KB row table)
#define BK_MAX_DYN_SMEM (220 * 1024)
#define BK_WPT 4            // bitmap words per thread at lbits = 16 (2048 words / 512 threads)

// bm[w].y = number of set presence bits below word w; returns the number of distinct k-mers.
// Ends with a barrier: bm is complete for every thread on return.
template <int NT>
__device__ __forceinline__ uint32_t bk_ranks(int nwords, uint2 *bm, uint32_t *s_wsum) {
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wpt = (nwords + NT - 1) / NT;   // 1 .. BK_WPT
    uint32_t loc[BK_WPT], cnt = 0;
#pragma unroll
    for (int j = 0; j < BK_WPT; j++) {
        const int w = (int)tid * wpt + j;
        loc[j] = (j < wpt && w < nwords) ? __popc(bm[w].x) : 0u;
        cnt += loc[j];
    }
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31) s_wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < NT / 32 ? s_wsum[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= (unsigned)o) wi += t;
        }
        if (lane < NT / 32) s_wsum[lane] = wi - w;
        if (lane == 31) s_wsum[32] = wi;
    }
    __syncthreads();
    uint32_t run = s_wsum[warp] + inc - cnt;
#pragma unroll
    for (int j = 0; j < BK_WPT; j++) {
        const int w = (int)tid * wpt + j;
        if (j < wpt && w < nwords) { bm[w].y = run; run += loc[j]; }
    }
    const uint32_t D = s_wsum[32];
    __syncthreads();
    return D;
}

// ---------------------------------------------------------------------------------------
// Paged variants (ps_paged.cuh): a bucket is a LIST of level-2 pages (<= 512 records each, 4-byte
// records low << 8 | sample & 255, the page carries the sample group). Warp w of a block takes pages w, w + NT/32,
// ...; a page (2 KB) is four coalesced 128-bit loads per lane, all independent, nothing shared between warps: no
// barriers and no shared-memory round trip. The pages are not staged in shared memory because the bucket kernels are
// shared-memory bound (bitmap tests and row atomics); a cp.async.bulk ring that staged them was measured slower.
// calls f(record, group) for every record of pages [0, npages) of one bucket; no barrier at the end.
template <int NT, typename F>
__device__ __forceinline__ void bk_for_each_direct(const unsigned long long *__restrict__ pages, uint32_t npages,
                                                   const uint32_t *__restrict__ recs_b, F f) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t p = warp; p < npages; p += NT / 32) {
        const unsigned long long e = __ldg(pages + p);
        const uint32_t cnt = BKP_CNT(e), grp = BKP_GRP(e);
        const uint4 *src = reinterpret_cast<const uint4 *>(recs_b + (size_t)BKP_PAGE(e) * PG_B);
        uint4 v[PG_B / 128];
#pragma unroll
        for (int j = 0; j < PG_B / 128; j++)
            v[j] = (uint32_t)(j * 128 + lane * 4) < cnt ? __ldg(src + j * 32 + lane) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int j = 0; j < PG_B / 128; j++) {
            const uint32_t i0 = j * 128 + lane * 4;
            if (i0 < cnt) f(v[j].x, grp);
            if (i0 + 1 < cnt) f(v[j].y, grp);
            if (i0 + 2 < cnt) f(v[j].z, grp);
            if (i0 + 3 < cnt) f(v[j].w, grp);
        }
    }
}

// order = the buckets with size[b] > big (from the front), then the others (from the back); size is the records of
// a bucket for k_bucket_count_pg and its distinct k-mers for k_bucket_build_pg. fill: two zeroed counters, and
// fill[0] ends as the number of big buckets.
__global__ void k_bucket_order_pg(const uint32_t *__restrict__ size, uint32_t big, uint32_t *__restrict__ fill,
                                  uint32_t *__restrict__ order) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= BK_N) return;                                 // BK_N is a multiple of 32: whole warps leave
    // one atomicAdd per warp and side: 65,536 single ones on two counters serialise
    const bool is_big = size[b] > big;
    const unsigned mbig = __ballot_sync(0xffffffffu, is_big), msmall = ~mbig, lt = lanemask_lt();
    uint32_t base_big = 0, base_small = 0;
    if ((threadIdx.x & 31) == 0) {
        if (mbig) base_big = atomicAdd(fill, (uint32_t)__popc(mbig));
        if (msmall) base_small = atomicAdd(fill + 1, (uint32_t)__popc(msmall));
    }
    base_big = __shfl_sync(0xffffffffu, base_big, 0);
    base_small = __shfl_sync(0xffffffffu, base_small, 0);
    const uint32_t pos = is_big ? base_big + __popc(mbig & lt) : (uint32_t)(BK_N - 1) - (base_small + __popc(msmall & lt));
    order[pos] = b;
}

__global__ void __launch_bounds__(BK_THREADS)
k_bucket_count_pg(const uint32_t *__restrict__ recs_b, const unsigned long long *__restrict__ blist,
                  const unsigned long long *__restrict__ bpstart, uint32_t G, const uint32_t *__restrict__ order, int lbits,
                  uint32_t *__restrict__ counts, uint32_t *__restrict__ gbm) {
    constexpr int NT = BK_THREADS;
    __shared__ uint32_t bits[BK_N / 32];
    __shared__ uint32_t s_part[NT / 32];
    const unsigned tid = threadIdx.x;
    const uint32_t b = order[blockIdx.x];
    const unsigned long long ps = bpstart[(size_t)b * G];
    const uint32_t npages = (uint32_t)(bpstart[(size_t)(b + 1) * G] - ps);
    if (npages == 0) { if (tid == 0) counts[b] = 0; return; }
    const int nwords = lbits >= 5 ? (1 << (lbits - 5)) : 1;
    for (int i = tid; i < nwords; i += NT) bits[i] = 0u;
    __syncthreads();
    const uint32_t lmask = (1u << lbits) - 1u;
    volatile uint32_t *vb = bits;
    // most records repeat a k-mer already seen in the bucket: test the bit before the atomic
    auto mark = [&](uint32_t rec, uint32_t) {
        const uint32_t low = (rec >> 8) & lmask;
        const uint32_t bit = 1u << (low & 31);
        if (!(vb[low >> 5] & bit)) atomicOr(&bits[low >> 5], bit);
    };
    bk_for_each_direct<NT>(blist + ps, npages, recs_b, mark);
    __syncthreads();
    uint32_t *g = gbm + (size_t)b * nwords;
    uint32_t cnt = 0;
    for (int i = tid; i < nwords; i += NT) {
        const uint32_t v = bits[i];
        g[i] = v;
        cnt += __popc(v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((tid & 31) == 0) s_part[tid >> 5] = cnt;
    __syncthreads();
    if (tid == 0) {
        uint32_t D = 0;
#pragma unroll
        for (int w = 0; w < NT / 32; w++) D += s_part[w];
        counts[b] = D;
    }
}

// Rows are assembled in shared memory one 256-sample COLUMN SLICE at a time (8 words per row; the pages of
// a bucket are listed by sample group, and a page's group is exactly that slice): a row of 5,000 samples is
// 640 bytes, far too wide to keep hundreds of them in shared memory, while a slice is 32 bytes — the table
// holds ~1,100 rows whatever N is. Every slice of every row is written exactly once (absent groups as zeros).
// dynamic shared memory: rows (row_cap_words) | bm (nwords uint2)
template <int NT>
__global__ void __launch_bounds__(NT)
k_bucket_build_pg(const uint32_t *__restrict__ recs_b, const unsigned long long *__restrict__ blist,
                  const unsigned long long *__restrict__ bpstart, uint32_t G, const uint32_t *__restrict__ order,
                  const unsigned long long *__restrict__ first_row, const uint32_t *__restrict__ gbm, int lbits, int wp,
                  uint32_t row_cap_words, uint64_t *__restrict__ union_out, uint32_t *__restrict__ matrix) {
    extern __shared__ __align__(8) uint32_t rows[];
    const int nwords = lbits >= 5 ? (1 << (lbits - 5)) : 1;
    uint2 *bm = reinterpret_cast<uint2 *>(rows + row_cap_words);
    __shared__ uint32_t s_wsum[33];
    const unsigned tid = threadIdx.x;
    const uint32_t b = order[blockIdx.x];
    const unsigned long long *bp = bpstart + (size_t)b * G;
    if (bp[G] == bp[0]) return;
    const unsigned long long base = first_row[b];
    const uint32_t D = (uint32_t)(first_row[b + 1] - base);
    if (D == 0) return;
    const uint32_t *g0 = gbm + (size_t)b * nwords;
    for (int i = tid; i < nwords; i += NT) bm[i] = make_uint2(g0[i], 0u);
    __syncthreads();
    bk_ranks<NT>(nwords, bm, s_wsum);
    const int wpt = (nwords + NT - 1) / NT;
#pragma unroll
    for (int j = 0; j < BK_WPT; j++) {
        const int w = (int)tid * wpt + j;
        if (j < wpt && w < nwords) {
            uint32_t bits = bm[w].x;
            unsigned long long r = base + bm[w].y;
            while (bits) {
                const int q = __ffs(bits) - 1;
                bits &= bits - 1;
                union_out[r++] = ((uint64_t)b << lbits) | (uint64_t)(w * 32 + q);
            }
        }
    }
    const uint32_t lmask = (1u << lbits) - 1u;
    const uint32_t gw_full = min((uint32_t)wp, 8u);               // words of a full slice
    const uint32_t stride = gw_full + 1u;                          // odd: a warp's 32 rows spread over all banks
    const uint32_t win = row_cap_words / stride;
    uint32_t *grow = matrix + base * (uint64_t)wp;
    // the table is cleared once; every pass clears the words it stores on its way out (one barrier and one
    // sweep of the table less per column slice)
    for (uint32_t i = tid; i < min(win, D) * stride; i += NT) rows[i] = 0u;
    __syncthreads();
    for (uint32_t r0 = 0; r0 < D; r0 += win) {
        const uint32_t nr = min(win, D - r0);
        for (uint32_t g = 0; g < G; g++) {
            const uint32_t gw = min(8u, (uint32_t)wp - 8u * g);   // the last slice may be narrower
            const uint32_t npages = (uint32_t)(bp[g + 1] - bp[g]);
            if (npages) {
                auto place = [&](uint32_t rec, uint32_t) {
                    const uint32_t low = (rec >> 8) & lmask;
                    const uint32_t s8 = rec & 255u;
                    const uint2 wv = bm[low >> 5];
                    const uint32_t row = wv.y + __popc(wv.x & ((1u << (low & 31)) - 1u)) - r0;
                    if (row < nr) atomicOr(rows + row * stride + (s8 >> 5), 1u << (s8 & 31));
                };
                bk_for_each_direct<NT>(blist + bp[g], npages, recs_b, place);
                __syncthreads();
            }
            uint32_t *gdst = grow + (uint64_t)r0 * wp + 8u * g;
            for (uint32_t i = tid; i < nr * gw; i += NT) {
                const uint32_t rr = i / gw, w = i - rr * gw;
                gdst[(uint64_t)rr * wp + w] = rows[rr * stride + w];
                rows[rr * stride + w] = 0u;
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------
// --kmerDB (modeling.py:367-372: `glistcompare -i` of the database list with the feature vector):
// keep the union k-mers that occur in the sorted database list `db`, and their matrix rows.
// One warp per 32 union rows: a binary search per row, ballot -> the warp's kept rows. WRITE = false
// counts them per warp (scanned by k_scan_sums / k_scan_chunks); WRITE = true copies k-mer and row to their new
// position, the lanes of the warp moving one row's words together.
template <bool WRITE>
__global__ void __launch_bounds__(256)
k_isect(const uint64_t *__restrict__ uni, uint64_t U, const uint64_t *__restrict__ db, uint64_t ndb,
        const uint32_t *__restrict__ matrix, int wp, uint32_t *__restrict__ warp_counts,
        const unsigned long long *__restrict__ warp_offs, uint64_t *__restrict__ uni_out, uint32_t *__restrict__ matrix_out) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t r = warp * 32 + lane;
    if (warp * 32 >= U) return;
    bool keep = false;
    uint64_t km = 0;
    if (r < U) {
        km = uni[r];
        uint64_t lo = 0, hi = ndb;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (__ldg(db + mid) < km) lo = mid + 1; else hi = mid;
        }
        keep = lo < ndb && __ldg(db + lo) == km;
    }
    const unsigned ball = __ballot_sync(0xffffffffu, keep);
    if (!WRITE) {
        if (lane == 0) warp_counts[warp] = __popc(ball);
        return;
    }
    const unsigned long long base = warp_offs[warp];
    if (keep) uni_out[base + __popc(ball & lanemask_lt())] = km;
    const uint32_t nk = __popc(ball);
    for (uint32_t i = lane; i < nk * (uint32_t)wp; i += 32) {
        const uint32_t j = i / wp, w = i - j * wp;
        const uint32_t src = __fns(ball, 0, j + 1);          // lane of the j-th kept row
        matrix_out[(base + j) * (uint64_t)wp + w] = matrix[(warp * 32 + src) * (uint64_t)wp + w];
    }
}

// Gather the matrix rows and k-mers of the survivors (slot order) for the D2H copy.
__global__ void k_gather_rows(const uint32_t *__restrict__ matrix, const uint64_t *__restrict__ uni,
                              const unsigned long long *__restrict__ sv_row, uint64_t ns, int wp,
                              uint32_t *__restrict__ out_bits, uint64_t *__restrict__ out_kmer) {
    const uint64_t total = ns * (uint64_t)wp;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s = i / wp;
        const uint32_t w = (uint32_t)(i % wp);
        const unsigned long long r = sv_row[s];
        out_bits[i] = matrix[r * (uint64_t)wp + w];
        if (w == 0) out_kmer[s] = uni[r];
    }
}
