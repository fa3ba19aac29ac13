// ps_paged.cuh — paged two-level partition of (k-mer, sample) instances: what regroups the
// sample-major k-mer instances of ALL samples into k-mer-major buckets for the matrix build.
//
// Replaces the merge tree of `glistcompare -u` and the N x U lookups of `glistquery -l`
// (modeling.py:317-380) for 16 < 2k <= 32 (k = 9..16: the k = 13 / 16 of the named configs).
//
// A k-mer (2k bits) = top16 (d2:8 | d1:8) | low (lbits = 2k - 16). Two scatter kernels bring the
// instances of one top16 value ("bucket") together; the bucket kernels (ps_rows.cuh) then resolve
// the low bits with a presence bitmap. Nothing is sorted and nothing is counted in advance:
//
//   k_scatter1  FUSED extraction + level-1 partition. A persistent block takes tiles of 8192
//               stream positions, computes the canonical k-mers, ranks them by bin = d2 + r
//               (r = destination GPU, from ascending k-mer splitters) with shared-memory atomics,
//               groups them in shared memory and APPENDS each bin's run to a PAGE that only this
//               block writes (1024 records; one open page per block and bin). A page that fills up
//               is closed (its meta word says which stream it belongs to and how many records it
//               holds) and a fresh one is taken from the pool with one atomicAdd. Because pages are
//               block-private there is no count pass, no global histogram, no look-back chain and
//               no ordering between blocks; invalid windows and out-of-range k-mers are simply not
//               written (compaction is free). The destination pool of a bin may be a PEER GPU's
//               memory (CUDA IPC mapping): the multi-GPU all-to-all is this kernel's write-out,
//               128-byte runs over NVLink.
//               Records are 4 bytes for any number of samples: d1 << 24 | low << 8 | (sample & 255);
//               the sample GROUP (sample >> 8) is a property of the page (a block closes its open
//               pages when the group of its tiles changes).
//   k_pga_*     tiny kernels: pages -> tiles of up to 8 pages of one stream (page ids and counts
//               in the tile descriptor).
//   k_scatter2  level-2 partition of every stream (group, bin) by d1 into pages of 512 records
//               tagged (bucket = d2 << 8 | d1, group). Input pages come in through the TMA unit
//               (cp.async.bulk global -> shared, mbarrier completion); closing a page also counts
//               it for its bucket's page list. The level-2 pages are the halves of the level-1 pages
//               the block has read (plus a small reserve): no second pool.
//   k_pgb_fill  pages -> per-bucket page lists (+ record counts for largest-first scheduling).
//
// The order of records inside a bucket is arbitrary (and varies from run to run); the bucket
// kernels OR presence bits, so union and matrix are deterministic.
#pragma once
#include "ps_common.cuh"
#include "ps_extract.cuh"

#define PG_A 1024            // records per level-1 page (4 KB)
#define PG_A_LOG 10
#define PG_B 512             // records per level-2 page (2 KB)
#define SC_THREADS 512
#define SC_ITEMS 16
#define SC_TILE (SC_THREADS * SC_ITEMS)      // 8192 positions / records per tile
#define SC_BINS1 264                          // 256 + PART_MAX - 1 bins at level 1, padded
#define SC_TILE_PAGES (SC_TILE / PG_A)        // level-2 tile = up to 8 level-1 pages
#define PG_NONE 0xFFFFFFFFu

// level-1 page meta (u32): stream key << 11 | count, key = group << 9 | bin; 0 = unused page
#define PGA_META(key, cnt) (((uint32_t)(key) << 11) | (uint32_t)(cnt))
#define PGA_KEY(m) ((m) >> 11)
#define PGA_CNT(m) ((m) & 2047u)
// level-2 page meta (u64): (bucket << 8 | group) << 32 | count; 0 = unused page
#define PGB_META(bucket, grp, cnt) ((((unsigned long long)(bucket) << 8 | (unsigned long long)(grp)) << 32) | (unsigned long long)(cnt))
// bucket page-list entry (u64): page | group << 32 | count << 40
#define BKP_ENTRY(page, grp, cnt) ((unsigned long long)(page) | ((unsigned long long)(grp) << 32) | ((unsigned long long)(cnt) << 40))
#define BKP_PAGE(e) ((uint32_t)(e))
#define BKP_GRP(e) ((uint32_t)((e) >> 32) & 255u)
#define BKP_CNT(e) ((uint32_t)((e) >> 40))

// One destination's page pool as a writer sees it. recs / meta belong to the pool's owner (this GPU
// or a peer); the writer owns pages [page0, page0 + cap) of it and counts them with a LOCAL cursor.
struct PgPool {
    uint32_t *recs;
    uint32_t *meta;
    uint32_t page0, cap;
};
struct Sc1Dst {
    PgPool pool[PART_MAX];
    uint32_t spl[PART_MAX];      // nparts - 1 ascending k-mer splitters (destination d owns [spl[d-1], spl[d]))
    int nparts;
    uint32_t *cursor;            // [PART_MAX] pages taken per destination (local)
    uint32_t *overflow;          // set to 1 when a sub-pool is exhausted (records then go to `trash`)
    uint32_t *trash;             // SC_TILE records of local scratch
};

// persistent per-block state of a scatter kernel: open page + fill per bin, current group / stream
struct ScState {
    uint32_t page[SC_BINS1];
    uint32_t fill[SC_BINS1];
    uint32_t spare[SC_BINS1];    // page taken ahead of need (PG_NONE = none)
    uint32_t key;                // level 1: group; level 2: stream key (group << 9 | bin)
    uint32_t pad[7];
};

// ---- mbarrier / bulk-copy (TMA) primitives -------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared through the TMA unit; bytes: multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- the shared back end of both scatter kernels ---------------------------------------------------
// Shared-memory working set of one block.
template <int NB>
struct ScShared {
    uint32_t cnt[2][NB + 8];                 // per-bin counts -> tile-local bases, cnt[NB] = records in the tile (double-buffered over tiles)
    uint32_t split[NB];                      // tile-local index where the run moves on to its second piece
    unsigned long long pab[NB][2];           // global address of tile-local index 0 for the run's piece A / piece B
    uint32_t wsum[SC_THREADS / 32];
    uint32_t next_tile;
};

// Block-wide exclusive scan of one value per bin (threads >= NB pass 0). Contains one barrier;
// the caller adds another before the results (cnt[] as cursors, pa/pb/split) are used.
template <int NB>
__device__ __forceinline__ uint32_t sc_bin_scan(uint32_t c, uint32_t *wsum) {
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t wp = 0;
#pragma unroll
    for (int w2 = 0; w2 < (NB + 31) / 32; w2++) if (w2 < (int)warp) wp += wsum[w2];
    return wp + inc - c;
}

// Write-out of the grouped tile in shared memory: thread t copies records t, t + 512, ... — consecutive
// lanes hold consecutive records of (mostly) one run, so a warp's store is one or two contiguous pieces.
// The bin of a record picks the run's page address; BINOF(record, index) supplies it.
template <int NB, typename BinOf, typename RecOf>
__device__ __forceinline__ void sc_write_flat(const uint32_t *sk, uint32_t total, const uint32_t *split,
                                              const unsigned long long (*pab)[2], BinOf bin_of, RecOf rec_of) {
#pragma unroll 4
    for (uint32_t p = threadIdx.x; p < total; p += SC_THREADS) {
        const uint32_t v = sk[p];
        const uint32_t b = bin_of(v, p);
        uint32_t *dst = reinterpret_cast<uint32_t *>(pab[b][p >= split[b] ? 1 : 0]);
        dst[p] = rec_of(v);
    }
}

// ---- level 1: extraction + scatter ------------------------------------------------------------------
// Page bookkeeping of bin `b` for a tile that holds c > 0 records of it starting at tile-local index
// tb. pool: where the bin's pages live. Sets pa/pb/split, updates the open page, closes full pages.
template <int PG, typename MetaFn>
__device__ __forceinline__ void sc_place_run(uint32_t c, uint32_t tb, uint32_t &pg, uint32_t &fill, uint32_t &spare,
                                             uint32_t *recs, uint32_t page0, uint32_t cap, uint32_t *cursor,
                                             uint32_t *overflow, uint32_t *trash, uint32_t &split,
                                             unsigned long long &pa, unsigned long long &pb, MetaFn close_page) {
    // one page: the spare taken ahead of need if there is one (its atomicAdd was issued many tiles ago,
    // so nothing waits here), else straight from the pool
    auto take = [&]() -> uint32_t {
        uint32_t r = spare;
        spare = PG_NONE;
        if (r == PG_NONE) {
            const uint32_t p = atomicAdd(cursor, 1u);
            if (p < cap) r = page0 + p;
        }
        return r;
    };
    if (pg == PG_NONE) { pg = take(); fill = 0; }
    if (pg != PG_NONE) {
        const uint32_t lenA = min(c, (uint32_t)PG - fill);
        pa = reinterpret_cast<unsigned long long>(recs + (size_t)pg * PG + fill) - 4ull * tb;
        split = tb + lenA;
        fill += lenA;
        if (fill == PG) { close_page(pg, (uint32_t)PG); pg = PG_NONE; fill = 0; }
        const uint32_t rest = c - lenA;
        pb = pa;
        if (rest) {
            // the remainder goes to freshly taken, CONSECUTIVE pages: one linear piece
            const uint32_t nnew = (rest + PG - 1) / PG;
            uint32_t first = PG_NONE;
            if (nnew == 1) first = take();
            else {
                const uint32_t p = atomicAdd(cursor, nnew);
                if (p + nnew <= cap) first = page0 + p;
            }
            if (first != PG_NONE) {
                pb = reinterpret_cast<unsigned long long>(recs + (size_t)first * PG) - 4ull * (tb + lenA);
                for (uint32_t q = 0; q + 1 < nnew; q++) close_page(first + q, (uint32_t)PG);
                const uint32_t tail = rest - (nnew - 1) * PG;
                if (tail == PG) { close_page(first + nnew - 1, (uint32_t)PG); }
                else { pg = first + nnew - 1; fill = tail; }
            } else {
                *overflow = 1u;
                pb = reinterpret_cast<unsigned long long>(trash) - 4ull * (tb + lenA);
            }
        }
        // half full: take the next page now, it will be needed in ~PG/64 tiles
        if (spare == PG_NONE && pg != PG_NONE && fill >= PG / 2) {
            const uint32_t p = atomicAdd(cursor, 1u);
            if (p < cap) spare = page0 + p;
        }
    } else {
        *overflow = 1u;
        split = tb + c;
        pa = reinterpret_cast<unsigned long long>(trash) - 4ull * tb;
        pb = pa;
    }
}

// Tiles of this launch: pool blocks (4096 positions) [blk0, blk0 + nblocks) taken two at a time.
// SRC 0: positions of the 2-bit stream pool; SRC 1: entries of the per-sample counted lists (u32 keys).
struct Sc1Src {
    const uint32_t *seq, *bad;        // SRC 0
    const uint32_t *list_keys;        // SRC 1
    const uint32_t *blk_valid;        // SRC 1: valid entries per list block (indexed from 0 at blk0)
    const uint16_t *blk_sample;       // sample of pool block b: blk_sample[b] (SRC 0: absolute block index; SRC 1: from 0 at blk0)
    uint64_t pos_begin;               // first position / entry (multiple of 4096)
    uint64_t nblocks;
    int k;
    uint32_t lo, hi;                  // k-mer range filter [lo, hi], inclusive hi (whole space: 0, 0xFFFFFFFF)
};

// Destination of level-1 bin b. A bin is one (d2, r) pair with b = d2 + r (r = destination = number of
// splitters <= the k-mer; pairs that can occur are ordered, so d2 + r is injective): find the r whose
// k-mer interval [spl[r-1], spl[r]) meets the interval of top byte d2 = b - r.
__device__ __forceinline__ int sc1_bin_dest(int b, const Sc1Dst &dst, int lbits) {
    for (int rr = 0; rr < dst.nparts; rr++) {
        const int d2 = b - rr;
        if (d2 < 0 || d2 > 255) continue;
        const uint32_t kmin = (uint32_t)d2 << (lbits + 8);
        const uint32_t kmax = kmin | ((1u << (lbits + 8)) - 1u);
        const uint32_t lo_s = rr ? dst.spl[rr - 1] : 0u;
        const bool last = rr == dst.nparts - 1;
        if (!last && dst.spl[rr] <= lo_s) continue;                      // empty interval
        if (kmax >= lo_s && (last || kmin < dst.spl[rr])) return rr;
    }
    return 0;
}

// destination of one k-mer: table lookup by top byte; only the (at most nparts - 1) top bytes whose
// interval holds a splitter need a compare
__device__ __forceinline__ uint32_t sc1_dest(uint32_t km, uint32_t d2, int nparts, const uint8_t *d2r, const uint32_t *spl) {
    if (nparts <= 1) return 0u;
    const uint32_t e = d2r[d2];
    uint32_t r = e & 15u;
    for (uint32_t j = e >> 4; j; j--) r += km >= spl[r] ? 1u : 0u;     // splitters ascend: stop mattering once one is larger
    return r;
}

// LEAN (stream source only): the k-mers are not kept in registers between the ranking and the grouping phase —
// phase A only counts the bins, phase C computes the window's k-mer again (four instructions from the word pair
// and its reversed complement) and takes its slot with an atomicAdd on the bin's base — so that 42 registers
// suffice and three blocks fit on an SM instead of two.
template <int SRC, bool LEAN>
__global__ void __launch_bounds__(SC_THREADS, LEAN ? 3 : 2)
k_scatter1(Sc1Src src, Sc1Dst dst, ScState *__restrict__ state, uint32_t *__restrict__ ticket) {
    constexpr int NB = SC_BINS1;
    extern __shared__ __align__(16) uint8_t sc_dyn[];
    uint32_t *sk = reinterpret_cast<uint32_t *>(sc_dyn);                       // SC_TILE records
    uint16_t *sb = reinterpret_cast<uint16_t *>(sc_dyn + SC_TILE * 4);         // their bins (the 32 record bits are all taken)
    ScShared<NB> &S = *reinterpret_cast<ScShared<NB> *>(sc_dyn + SC_TILE * 6);
    __shared__ uint32_t s_spl[PART_MAX];
    __shared__ uint32_t s_group;
    __shared__ uint8_t s_binr[NB];
    __shared__ uint8_t s_d2r[256];       // per top byte d2: destination of its smallest k-mer | splitters inside its interval << 4
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = src.k, lbits = 2 * k - 16;
    const uint32_t lowmask = (1u << lbits) - 1u;               // the bits below the two top bytes d2, d1
    const int nparts = dst.nparts;
    ScState &st = state[blockIdx.x];
    // thread b < NB owns bin b for the whole kernel: open page, fill and spare page live in registers
    uint32_t my_pg = PG_NONE, my_fill = 0, my_spare = PG_NONE;
    if (tid < NB) { my_pg = st.page[tid]; my_fill = st.fill[tid]; my_spare = st.spare[tid]; S.cnt[0][tid] = 0; S.cnt[1][tid] = 0; }
    if (tid < PART_MAX) s_spl[tid] = (int)tid < nparts - 1 ? dst.spl[tid] : 0xFFFFFFFFu;
    if (tid < NB) s_binr[tid] = (uint8_t)sc1_bin_dest((int)tid, dst, lbits);
    if (tid < 256) {
        const uint32_t kmin = tid << (lbits + 8), kmax = kmin | ((1u << (lbits + 8)) - 1u);
        uint32_t r0 = 0, nin = 0;
        for (int p = 0; p < nparts - 1; p++) {
            if (dst.spl[p] <= kmin) r0++;
            else if (dst.spl[p] <= kmax) nin++;
        }
        s_d2r[tid] = (uint8_t)(r0 | (nin << 4));
    }
    if (tid == 0) { s_group = st.key; S.next_tile = atomicAdd(ticket, 1u); }
    __syncthreads();
    const uint32_t ntiles = (uint32_t)((src.nblocks + 1) / 2);
    uint32_t tile = S.next_tile;
    int buf = 0;
    while (tile < ntiles) {
        const uint64_t b0 = 2ull * tile;
        const int nb = (int)min((uint64_t)2, src.nblocks - b0);
        const uint64_t tb0 = (SRC == 0 ? (src.pos_begin >> 12) : 0ull) + b0;
        const uint32_t tagA = src.blk_sample[tb0], tagB = nb == 2 ? src.blk_sample[tb0 + 1] : tagA;
        const int nsub = (tagA >> 8) != (tagB >> 8) ? 2 : 1;     // a tile never mixes sample groups
        for (int sub = 0; sub < nsub; sub++) {
            uint32_t *cnt = S.cnt[buf], *cnt_next = S.cnt[buf ^ 1];
            const unsigned half = warp >> 3;                     // warps 0-7: first block of the tile, 8-15: second
            const bool on = (int)half < nb && (nsub == 1 || (int)half == sub);
            const uint32_t tag8 = (half ? tagB : tagA) & 255u;
            const uint32_t group = (nsub == 2 && sub == 1) ? (tagB >> 8) : (tagA >> 8);
            // ---- A: canonical k-mers of my 16 positions, ranked inside their bin ----
            uint32_t km[LEAN ? 1 : SC_ITEMS];
            uint32_t rk[LEAN ? 1 : SC_ITEMS / 2];                // two 16-bit ranks per register
            uint32_t vmask = 0;
            uint32_t lw0 = 0, lw1 = 0, lrc_hi = 0, lrc_lo = 0;  // LEAN: what phase C needs to compute the k-mers again
            if (on) {
                const uint64_t local = (b0 << 12) + (uint64_t)warp * 512;       // warp's 512 positions
                if (SRC == 0) {
                    // Lane l owns the 16 CONSECUTIVE positions 16 l .. 16 l + 15 of the warp's 512: they start
                    // exactly at sequence word l, and a window of k <= 16 bases reaches at most into word l + 1
                    // (one shuffle per lane instead of four per k-mer); the 32 mask bits from position 16 l on
                    // come from mask words l/2 and l/2 + 1. The order of records inside a tile is free.
                    const uint64_t base = src.pos_begin + local;
                    const uint64_t wbase = base >> 4;
                    const uint32_t w0 = __ldg(src.seq + wbase + lane);
                    const uint32_t wext = __ldg(src.seq + wbase + 32);
                    uint32_t w1 = __shfl_down_sync(0xffffffffu, w0, 1);
                    if (lane == 31) w1 = wext;
                    const uint32_t myb = __ldg(src.bad + (base >> 5) + min(lane, 16u));
                    const uint32_t m0 = __shfl_sync(0xffffffffu, myb, lane >> 1), m1 = __shfl_sync(0xffffffffu, myb, (lane >> 1) + 1);
                    const uint32_t badwin = __funnelshift_r(m0, m1, 16u * (lane & 1u));
                    const uint32_t kmask = (1u << k) - 1u;
                    const uint32_t dn = 32 - 2 * k;
                    // Reverse complement of the lane's 32 bases ONCE (two BREV-based word reversals); the reverse
                    // complement of the window at position `it` is then bases 32-it-k .. 31-it of it: one funnel
                    // shift by a compile-time amount after a common pre-shift by 34 - 2k bits.
                    const uint64_t rcw = (((uint64_t)rev2_32(~w1) << 32) | (uint64_t)rev2_32(~w0)) << (34 - 2 * k);
                    const uint32_t rc_hi = (uint32_t)(rcw >> 32), rc_lo = (uint32_t)rcw;
                    const uint32_t span = src.hi - src.lo;
#pragma unroll
                    for (int it = 0; it < SC_ITEMS; it++) {
                        const uint32_t fw = __funnelshift_l(w1, w0, 2 * it) >> dn;
                        const uint32_t rc = __funnelshift_l(rc_lo, rc_hi, 30 - 2 * it) >> dn;
                        const uint32_t key = fw < rc ? fw : rc;
                        const bool ok = ((badwin >> it) & kmask) == 0 && key - src.lo <= span;
                        if (LEAN) {
                            if (ok) {
                                const uint32_t d2 = key >> (lbits + 8);
                                atomicAdd(&cnt[d2 + sc1_dest(key, d2, nparts, s_d2r, s_spl)], 1u);
                            }
                        } else km[it] = key;
                        vmask |= (ok ? 1u : 0u) << it;
                    }
                    if (LEAN) { lw0 = w0; lw1 = w1; lrc_hi = rc_hi; lrc_lo = rc_lo; }
                } else {
                    const uint32_t nvalid = src.blk_valid[b0 + half];
                    const uint32_t *lk = src.list_keys + src.pos_begin + local;
#pragma unroll
                    for (int it = 0; it < SC_ITEMS; it++) {
                        const uint32_t li = (warp & 7) * 512 + it * 32 + lane;
                        const bool in = li < nvalid;
                        const uint32_t key = in ? lk[it * 32 + lane] : 0u;
                        km[it] = key;
                        vmask |= ((in && key >= src.lo && key <= src.hi) ? 1u : 0u) << it;
                    }
                }
                if (!LEAN) {
#pragma unroll
                    for (int it = 0; it < SC_ITEMS; it++) {
                        uint32_t rnk = 0;
                        if ((vmask >> it) & 1u) {
                            const uint32_t d2 = km[LEAN ? 0 : it] >> (lbits + 8);
                            rnk = atomicAdd(&cnt[d2 + sc1_dest(km[LEAN ? 0 : it], d2, nparts, s_d2r, s_spl)], 1u);
                        }
                        if (it & 1) rk[LEAN ? 0 : it >> 1] |= rnk << 16; else rk[LEAN ? 0 : it >> 1] = rnk;
                    }
                }
            }
            __syncthreads();
            // ---- B: bins -> tile-local bases, page bookkeeping; next ticket ----
            if (tid == 0 && sub == nsub - 1) S.next_tile = atomicAdd(ticket, 1u);
            const uint32_t c = tid < NB ? cnt[tid] : 0u;
            const uint32_t tb = sc_bin_scan<NB>(c, S.wsum);
            if (tid < NB) {
                cnt[tid] = tb;
                if (tid == NB - 1) cnt[NB] = tb + c;
                cnt_next[tid] = 0;
                const int r = s_binr[tid];
                const PgPool &P = dst.pool[r];
                if (group != s_group && my_pg != PG_NONE) {       // tiles moved on to another sample group
                    if (my_fill) P.meta[my_pg] = PGA_META((s_group << 9) | tid, my_fill);
                    my_pg = PG_NONE; my_fill = 0;
                }
                if (c) {
                    const uint32_t key = (group << 9) | tid;
                    uint32_t *meta = P.meta;
                    sc_place_run<PG_A>(c, tb, my_pg, my_fill, my_spare, P.recs, P.page0, P.cap, dst.cursor + r, dst.overflow,
                                       dst.trash, S.split[tid], S.pab[tid][0], S.pab[tid][1],
                                       [meta, key](uint32_t page, uint32_t n) { meta[page] = PGA_META(key, n); });
                }
            }
            __syncthreads();
            if (tid == 0) s_group = group;
            // the words of the NEXT tile (its ticket is known since phase B) start their way into L2 now: the
            // first thing a tile does is wait for them (24 % of the stall samples sat on that load)
            if (SRC == 0 && sub == nsub - 1) {
                const uint32_t nt = S.next_tile;
                if (nt < ntiles && (int)(warp >> 3) < (int)min((uint64_t)2, src.nblocks - (uint64_t)2 * nt)) {
                    const uint64_t nbase = src.pos_begin + ((2ull * nt) << 12) + (uint64_t)warp * 512;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(src.seq + (nbase >> 4) + lane));
                    if (lane <= 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(src.bad + (nbase >> 5) + lane));
                }
            }
            // ---- C: group the records in shared memory ----
            if (on) {
                const uint32_t dn = 32 - 2 * k;
#pragma unroll
                for (int it = 0; it < SC_ITEMS; it++) {
                    if ((vmask >> it) & 1u) {
                        uint32_t key;
                        if (LEAN) {
                            const uint32_t fw = __funnelshift_l(lw1, lw0, 2 * it) >> dn;
                            const uint32_t rc = __funnelshift_l(lrc_lo, lrc_hi, 30 - 2 * it) >> dn;
                            key = fw < rc ? fw : rc;
                        } else key = km[LEAN ? 0 : it];
                        const uint32_t d2 = key >> (lbits + 8);
                        const uint32_t bin = d2 + sc1_dest(key, d2, nparts, s_d2r, s_spl);
                        // LEAN: cnt[bin] holds the bin's base and moves up with every record placed (the order
                        // inside a bin is free); otherwise base + the rank taken in phase A
                        const uint32_t pos = LEAN ? atomicAdd(&cnt[bin], 1u)
                                                  : cnt[bin] + ((it & 1) ? (rk[LEAN ? 0 : it >> 1] >> 16) : (rk[LEAN ? 0 : it >> 1] & 0xFFFFu));
                        // d1 << 24 | low << 8 | sample & 255 (low has lbits <= 16 bits: d1 sits at bit 24 for every k)
                        sk[pos] = (((key >> lbits) & 255u) << 24) | ((key & lowmask) << 8) | tag8;
                        sb[pos] = (uint16_t)bin;
                    }
                }
            }
            __syncthreads();
            // ---- D: runs -> pages ----
            sc_write_flat<NB>(sk, cnt[NB], S.split, S.pab, [sb](uint32_t, uint32_t p) { return (uint32_t)sb[p]; },
                              [](uint32_t v) { return v; });
            __syncthreads();
            buf ^= 1;
        }
        tile = S.next_tile;
    }
    if (tid < NB) { st.page[tid] = my_pg; st.fill[tid] = my_fill; st.spare[tid] = my_spare; }
    if (tid == 0) st.key = s_group;
}

// Closes the open pages of every block state (writes their meta) and resets the state.
// LEVEL 1: the pool of bin b is found like in k_scatter1; LEVEL 2: one local pool, u64 meta.
__global__ void k_pg_close1(ScState *__restrict__ state, Sc1Dst dst, int lbits) {
    const unsigned tid = threadIdx.x;
    ScState &st = state[blockIdx.x];
    const uint32_t group = st.key;
    __syncthreads();                       // everybody has the group before thread 0 resets it
    if (tid < SC_BINS1) {
        const uint32_t pg = st.page[tid], fill = st.fill[tid];
        if (pg != PG_NONE && fill) {
            const int r = sc1_bin_dest((int)tid, dst, lbits);
            dst.pool[r].meta[pg] = PGA_META((group << 9) | tid, fill);
        }
        const uint32_t sp = st.spare[tid];
        if (sp != PG_NONE) dst.pool[sc1_bin_dest((int)tid, dst, lbits)].meta[sp] = 0u;     // taken ahead of need, never used
        st.page[tid] = PG_NONE;
        st.fill[tid] = 0;
        st.spare[tid] = PG_NONE;
    }
    if (tid == 0) st.key = 0;
}

__global__ void k_pg_reset_state(ScState *__restrict__ state) {
    const unsigned tid = threadIdx.x;
    ScState &st = state[blockIdx.x];
    if (tid < SC_BINS1) { st.page[tid] = PG_NONE; st.fill[tid] = 0; st.spare[tid] = PG_NONE; }
    if (tid == 0) st.key = 0;
}

// ---- level-1 pages -> stream page lists -> level-2 tiles ---------------------------------------------
// Single block: exclusive scan of the tile counts ceil(scnt / 8) (-> tstart, ns + 1 entries; tstart[ns] = tiles).
// sfill is zeroed.
__global__ void __launch_bounds__(1024)
k_pga_scan(const uint32_t *__restrict__ scnt, uint32_t ns, uint32_t *__restrict__ tstart,
           uint32_t *__restrict__ sfill) {
    __shared__ uint32_t ws[32];
    __shared__ uint32_t carry;
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < ns; base += 1024) {
        const uint32_t i = base + tid;
        const uint32_t b = i < ns ? (scnt[i] + SC_TILE_PAGES - 1) / SC_TILE_PAGES : 0u;
        uint32_t ib = b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, ib, o);
            if (lane >= (unsigned)o) ib += t;
        }
        if (lane == 31) ws[warp] = ib;
        __syncthreads();
        if (warp == 0) {
            const uint32_t w = ws[lane];
            uint32_t x = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= (unsigned)o) x += t;
            }
            ws[lane] = x - w;
        }
        __syncthreads();
        const uint32_t e = carry + ws[warp] + ib - b;
        if (i < ns) { tstart[i] = e; sfill[i] = 0; }
        __syncthreads();
        if (tid == 1023) carry = e + b;
        __syncthreads();
    }
    if (tid == 0) tstart[ns] = carry;
}

// One level-2 tile: up to SC_TILE_PAGES level-1 pages of one stream, with their record counts, so that k_scatter2
// starts the copies of a tile after a single load.
struct __align__(16) Sc2Tile {
    uint32_t key, np;                    // stream key (group << 9 | bin), pages in the tile
    uint32_t page[SC_TILE_PAGES];
    uint16_t cnt[SC_TILE_PAGES];
    uint32_t pad[2];
};

// Page counts per stream (FILL = false: scnt[key] += pages) and tiles (FILL = true: page p, the j-th page of its
// stream in any order, goes to slot j % 8 of the stream's tile j / 8). A block takes PGL_THREADS x PGL_PER consecutive
// pages and adds them up per stream key in shared memory first (slot = key mod PGL_SLOTS; a page whose slot another
// key already holds goes to global memory on its own): one global atomicAdd per key and block instead of one per page.
// Consecutive pages were taken at about the same time, so they belong to a few dozen keys; the keys of a range
// share a few cache lines of scnt / sfill, and single atomics on them serialise (1 ms per launch on config 5).
// Only pages of level-1 bins [bin_lo, bin_hi) are listed: a build may cover a sub-range of the k-mer range
// the pool was scattered for (bins ascend with the k-mer), see ps_scatter_range.
#define PGL_THREADS 256
#define PGL_PER 8
#define PGL_SLOTS 2048
template <bool FILL>
__global__ void __launch_bounds__(PGL_THREADS)
k_pga_pages(const uint32_t *__restrict__ meta, uint32_t npages, uint32_t bin_lo, uint32_t bin_hi,
            uint32_t *__restrict__ scnt, const uint32_t *__restrict__ tstart, uint32_t *__restrict__ sfill,
            Sc2Tile *__restrict__ tiles) {
    __shared__ uint32_t s_tag[PGL_SLOTS], s_cnt[PGL_SLOTS];
    const unsigned tid = threadIdx.x;
    for (uint32_t i = tid; i < PGL_SLOTS; i += PGL_THREADS) { s_tag[i] = PG_NONE; s_cnt[i] = 0; }
    __syncthreads();
    const uint32_t p0 = blockIdx.x * (PGL_THREADS * PGL_PER) + tid;
    uint32_t m[PGL_PER], rank[PGL_PER];                // rank inside the block's pages of the key; PG_NONE: on its own
#pragma unroll
    for (int j = 0; j < PGL_PER; j++) {
        const uint32_t p = p0 + j * PGL_THREADS;
        m[j] = p < npages ? meta[p] : 0u;
        const uint32_t key = PGA_KEY(m[j]);
        if (!m[j] || (key & 511u) < bin_lo || (key & 511u) >= bin_hi) { m[j] = 0; continue; }
        const uint32_t slot = key & (PGL_SLOTS - 1);
        uint32_t tag = s_tag[slot];
        if (tag == PG_NONE) {
            tag = atomicCAS(&s_tag[slot], PG_NONE, key);
            if (tag == PG_NONE) tag = key;
        }
        rank[j] = tag == key ? atomicAdd(&s_cnt[slot], 1u) : PG_NONE;
        if (!FILL && rank[j] == PG_NONE) atomicAdd(&scnt[key], 1u);
    }
    __syncthreads();
    // one global atomicAdd per key; FILL: s_cnt[slot] becomes the index of the slot's first page in its stream
    for (uint32_t i = tid; i < PGL_SLOTS; i += PGL_THREADS) {
        const uint32_t c = s_cnt[i];
        if (!c) continue;
        const uint32_t b = atomicAdd(FILL ? &sfill[s_tag[i]] : &scnt[s_tag[i]], c);
        if (FILL) s_cnt[i] = b;
    }
    if (!FILL) return;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PGL_PER; j++) {
        if (!m[j]) continue;
        const uint32_t key = PGA_KEY(m[j]);
        const uint32_t idx = rank[j] == PG_NONE ? atomicAdd(&sfill[key], 1u) : s_cnt[key & (PGL_SLOTS - 1)] + rank[j];
        const uint32_t q = idx % SC_TILE_PAGES;
        Sc2Tile &t = tiles[tstart[key] + idx / SC_TILE_PAGES];
        t.page[q] = p0 + j * PGL_THREADS;
        t.cnt[q] = (uint16_t)PGA_CNT(m[j]);
        if (q == 0) { t.key = key; t.np = min((uint32_t)SC_TILE_PAGES, scnt[key] - idx); }
    }
}

// ---- level 2: pages of one stream -> pages of its 256 buckets ----------------------------------------
// Level-2 pages (2 KB) live in the level-1 buffer: slots 2p and 2p + 1 are the two halves of level-1 page p, and the
// `nres` slots from res0 = 2 x (level-1 pages) on are a reserve that the level-1 cursor never hands out. k_scatter2
// reads every level-1 page of a range exactly once; when the copy of a tile has completed, the tile's pages are dead
// and their slots join the SUPPLY of the block that read them. A block takes its pages from its own supply first, so
// only the block that read a page ever writes it, and no separate level-2 pool is needed.
//
// Reserve bound. The records of a block's tiles up to tile t fill at most two slots per level-1 page of those tiles,
// and that is what its supply has received by then. Beyond that the block holds at most 256 open pages, and every
// change of stream closes at most 256 partial pages. A block changes stream at most once per stream of its tile
// interval, so over all blocks demand beyond supply is at most (streams + 2 x blocks) x 256 pages, with streams <=
// G x SC_BINS1 (a level-1 stream is a (group, bin) pair): one term for the stream a block shares with its neighbour,
// one for the open pages at the end. The supply ring drops slots only while it holds SC2_FREE >= 256 + 16 of them;
// whatever the block is short of afterwards is again covered by its stream changes. The overflow flag stays as a check.
struct Sc2Args {
    uint32_t *recs;                      // level-1 pool (this GPU's own) and, in the same bytes, the level-2 slots
    const Sc2Tile *tiles;
    const uint32_t *ntiles;              // device scalar: tstart[ns]
    const uint8_t *bin_d2;               // [SC_BINS1] bin -> d2 for the bins this GPU owns
    unsigned long long *meta_b;          // per level-2 slot
    uint32_t res0, nres;                 // reserve slots [res0, res0 + nres)
    uint32_t *cursor_b;                  // reserve slots taken
    uint32_t *overflow;
    uint32_t *trash;
    uint32_t *bpcnt, *brecs;             // [BK_N * G] pages per (bucket, group), [BK_N] records per bucket
    uint32_t G;
};

// Closes level-2 page `page` (n records of bucket, group) and counts it for the bucket page lists.
__device__ __forceinline__ void pgb_close(unsigned long long *meta_b, uint32_t *bpcnt, uint32_t *brecs, uint32_t G,
                                          uint32_t page, uint32_t bucket, uint32_t grp, uint32_t n) {
    meta_b[page] = PGB_META(bucket, grp, n);
    atomicAdd(&bpcnt[bucket * G + grp], 1u);
    atomicAdd(&brecs[bucket], n);
}

// 8192-record tiles through ONE landing zone, three blocks per SM (40 registers). Phase A only counts the bins,
// phase C reads each record from the landing zone again and takes its slot with an atomicAdd on the bin's base; the
// copy of tile t + 1 starts once phase C has read the zone, and the other blocks on the SM cover the wait.
// (Two landing zones of 4096 records at four blocks per SM, ranks kept in registers: 124 vs 81 ms on config 5.)
#define SC2_BLOCKS_PER_SM 3
#define SC2_SMEM (2 * SC_TILE * 4 + sizeof(ScShared<256>))
#define SC2_FREE 512                     // supply ring of a block: >= 256 open pages + the 16 slots of one tile
#define SC2_XPG 32                       // pages of the runs longer than one page in one tile: <= 8192 / 512 + 15

// One level-2 page: the oldest free slot of the block's supply (ring[head, tail)), else a reserve slot.
__device__ __forceinline__ uint32_t sc2_take(const Sc2Args &a, const uint32_t *ring, uint32_t *head, uint32_t tail) {
    const uint32_t h = atomicAdd(head, 1u);
    if (h < tail) return ring[h & (SC2_FREE - 1)];
    const uint32_t r = atomicAdd(a.cursor_b, 1u);
    return r < a.nres ? a.res0 + r : PG_NONE;
}

// Page bookkeeping of bin `b` for a tile that holds c > 0 records of it starting at tile-local index tb: like
// sc_place_run, except that pages come one at a time and need not be adjacent. A remainder longer than one page is
// described by its page addresses in xpg[x ..] (pb = x << 1 | 1; a page address is even).
template <typename CloseFn>
__device__ __forceinline__ void sc2_place_run(const Sc2Args &a, uint32_t c, uint32_t tb, uint32_t &pg, uint32_t &fill,
                                              const uint32_t *ring, uint32_t *head, uint32_t tail, unsigned long long *xpg,
                                              uint32_t *nx, uint32_t &split, unsigned long long &pa, unsigned long long &pb,
                                              CloseFn close_page) {
    auto addr = [&](uint32_t slot) -> unsigned long long {
        return reinterpret_cast<unsigned long long>(slot == PG_NONE ? a.trash : a.recs + (size_t)slot * PG_B);
    };
    if (pg == PG_NONE) { pg = sc2_take(a, ring, head, tail); fill = 0; }
    if (pg == PG_NONE) {
        *a.overflow = 1u;
        split = tb + c;
        pa = pb = addr(PG_NONE) - 4ull * tb;
        return;
    }
    const uint32_t lenA = min(c, (uint32_t)PG_B - fill);
    pa = addr(pg) + 4ull * fill - 4ull * tb;
    split = tb + lenA;
    fill += lenA;
    if (fill == PG_B) { close_page(pg, (uint32_t)PG_B); pg = PG_NONE; fill = 0; }
    const uint32_t rest = c - lenA;
    pb = pa;
    if (!rest) return;
    const uint32_t nnew = (rest + PG_B - 1) / PG_B;
    const uint32_t x = nnew > 1 ? atomicAdd(nx, nnew) : 0u;
    for (uint32_t q = 0; q < nnew; q++) {
        const uint32_t s = sc2_take(a, ring, head, tail);
        if (s == PG_NONE) *a.overflow = 1u;
        if (nnew > 1) xpg[x + q] = addr(s);
        else pb = addr(s) - 4ull * (tb + lenA);
        const uint32_t n = min(rest - q * PG_B, (uint32_t)PG_B);
        if (s != PG_NONE) {
            if (n == PG_B) close_page(s, (uint32_t)PG_B);
            else { pg = s; fill = n; }
        }
    }
    if (nnew > 1) pb = (unsigned long long)x << 1 | 1ull;
}

__global__ void __launch_bounds__(SC_THREADS, SC2_BLOCKS_PER_SM)
k_scatter2(Sc2Args a, ScState *__restrict__ state) {
    constexpr int NB = 256;
    extern __shared__ __align__(128) uint8_t sc2_dyn[];
    uint32_t *sin = reinterpret_cast<uint32_t *>(sc2_dyn);                      // SC_TILE records (TMA landing zone)
    uint32_t *sk = sin + SC_TILE;                                               // SC_TILE records
    ScShared<NB> &S = *reinterpret_cast<ScShared<NB> *>(sc2_dyn + 2 * SC_TILE * 4);
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t s_pcnt[SC_TILE_PAGES];
    __shared__ uint32_t s_tpage[SC_TILE_PAGES];                     // level-1 pages of the tile in the landing zone
    __shared__ uint32_t s_key;
    __shared__ uint32_t s_cur_key;
    __shared__ Sc2Tile s_next;                                      // descriptor of the next tile to copy in
    __shared__ uint32_t s_ring[SC2_FREE];                           // the block's supply: free slots [s_head, s_tail)
    __shared__ uint32_t s_head, s_tail, s_nx;
    __shared__ unsigned long long s_xpg[SC2_XPG];
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    ScState &st = state[blockIdx.x];
    const uint32_t T = *a.ntiles;
    const uint32_t t_lo = (uint32_t)((uint64_t)T * blockIdx.x / gridDim.x), t_hi = (uint32_t)((uint64_t)T * (blockIdx.x + 1) / gridDim.x);
    uint32_t my_pg = PG_NONE, my_fill = 0;                          // thread b < 256 owns bin b
    if (tid < NB) { S.cnt[0][tid] = 0; S.cnt[1][tid] = 0; }
    if (tid == 0) {
        s_cur_key = 0;
        s_head = 0; s_tail = 0; s_nx = 0;
        mbar_init(&bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    // Warp 0 feeds the TMA unit. The descriptor of the next tile comes into shared memory by cp.async a whole tile
    // ahead, so that no load waits when the copies start; lane j < SC_TILE_PAGES copies page j.
    auto fetch = [&](uint32_t t) {
        if (lane < sizeof(Sc2Tile) / 16 && t < t_hi)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(reinterpret_cast<uint4 *>(&s_next) + lane)),
                         "l"(reinterpret_cast<const uint4 *>(a.tiles + t) + lane) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto issue = [&]() {
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
        const uint32_t c = lane < SC_TILE_PAGES && lane < s_next.np ? (uint32_t)s_next.cnt[lane] : 0u;
        const uint32_t bytes = (c * 4 + 15) & ~15u;
        const uint32_t total = __reduce_add_sync(0xffffffffu, bytes);
        if (lane < SC_TILE_PAGES) { s_pcnt[lane] = c; s_tpage[lane] = s_next.page[lane]; }
        if (lane == 0) { s_key = s_next.key; mbar_expect_tx(&bar, total); }
        __syncwarp();
        if (bytes) bulk_g2s(sin + lane * PG_A, a.recs + (size_t)s_next.page[lane] * PG_A, bytes, &bar);
        __syncwarp();                                               // s_next has been read: the next fetch may land
    };
    if (warp == 0 && t_lo < t_hi) {
        fetch(t_lo);
        issue();
    }
    uint32_t phase = 0;                                            // parity to wait for on the landing zone
    int buf = 0;
    for (uint32_t t = t_lo; t < t_hi; t++, buf ^= 1) {
        uint32_t *cnt = S.cnt[buf], *cnt_next = S.cnt[buf ^ 1];
        mbar_wait(&bar, phase);
        phase ^= 1u;
        if (warp == 0) {
            // The tile's pages have been read: their slots join the supply. No proxy fence is needed before the generic
            // stores that will reuse these bytes: the complete_tx that ended the wait comes after the bulk copy has read
            // its source, and the completion of a bulk copy carries an implicit generic-async proxy fence (PTX ISA,
            // cp.async.bulk). A slot's meta is cleared here, so that a slot that is never used lists nothing.
            const bool v = lane < 2 * SC_TILE_PAGES && s_pcnt[lane >> 1] != 0;
            const uint32_t nslot = __popc(__ballot_sync(0xffffffffu, v));
            const uint32_t tail = s_tail, room = SC2_FREE - (tail - s_head);
            if (v) {
                const uint32_t slot = 2 * s_tpage[lane >> 1] + (lane & 1u);
                a.meta_b[slot] = 0ull;
                if (lane < room) s_ring[(tail + lane) & (SC2_FREE - 1)] = slot;
            }
            __syncwarp();
            if (lane == 0) s_tail = tail + min(nslot, room);
            fetch(t + 1);
        }
        // ---- A: count the records of every bin (one shared-memory atomic per record) ----
#pragma unroll
        for (int it = 0; it < SC_ITEMS; it++) {
            const uint32_t i = it * SC_THREADS + tid;
            if ((i & (PG_A - 1)) < s_pcnt[i >> PG_A_LOG]) atomicAdd(&cnt[sin[i] >> 24], 1u);
        }
        __syncthreads();
        // ---- B: bins -> tile-local bases, page bookkeeping ----
        const uint32_t c = tid < NB ? cnt[tid] : 0u;
        const uint32_t tb = sc_bin_scan<NB>(c, S.wsum);
        const uint32_t key = s_key;
        if (tid < NB) {
            cnt[tid] = tb;
            if (tid == NB - 1) cnt[NB] = tb + c;
            cnt_next[tid] = 0;
            const uint32_t ckey = s_cur_key;
            if (key != ckey && my_pg != PG_NONE) {                 // the block moved on to another stream
                if (my_fill) pgb_close(a.meta_b, a.bpcnt, a.brecs, a.G, my_pg, ((uint32_t)a.bin_d2[ckey & 511u] << 8) | tid, ckey >> 9, my_fill);
                my_pg = PG_NONE; my_fill = 0;
            }
            if (c) {
                const uint32_t bucket = ((uint32_t)a.bin_d2[key & 511u] << 8) | tid, grp = key >> 9;
                unsigned long long *meta = a.meta_b;
                uint32_t nfull = 0;                                // pages sc2_place_run closes are full
                sc2_place_run(a, c, tb, my_pg, my_fill, s_ring, &s_head, s_tail, s_xpg, &s_nx, S.split[tid], S.pab[tid][0],
                              S.pab[tid][1], [meta, bucket, grp, &nfull](uint32_t page, uint32_t n) { meta[page] = PGB_META(bucket, grp, n); nfull++; });
                if (nfull) {
                    atomicAdd(&a.bpcnt[bucket * a.G + grp], nfull);
                    atomicAdd(&a.brecs[bucket], nfull * PG_B);
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            s_cur_key = key;
            if (s_head > s_tail) s_head = s_tail;                  // takes past the end went to the reserve
            s_nx = 0;
        }
        // ---- C: group the records in shared memory ----
        // cnt[bin] holds the bin's base and moves up with every record placed (the order inside a bin is free). The
        // volatile reads make this a second read of shared memory, not phase A's values kept in (spilled) registers.
#pragma unroll
        for (int it = 0; it < SC_ITEMS; it++) {
            const uint32_t i = it * SC_THREADS + tid;
            if ((i & (PG_A - 1)) < reinterpret_cast<const volatile uint32_t *>(s_pcnt)[i >> PG_A_LOG]) {
                const uint32_t r = reinterpret_cast<const volatile uint32_t *>(sin)[i];
                sk[atomicAdd(&cnt[r >> 24], 1u)] = r;               // the top byte (bin) is dropped on the way out
            }
        }
        __syncthreads();
        // the landing zone has been read: the next tile comes in during the write-out
        if (warp == 0 && t + 1 < t_hi) issue();
        // ---- D: runs -> pages (a run's piece B either linear or, longer than a page, through s_xpg) ----
        const uint32_t total = cnt[NB];
#pragma unroll 4
        for (uint32_t p = tid; p < total; p += SC_THREADS) {
            const uint32_t v = sk[p], b = v >> 24, sp = S.split[b];
            const unsigned long long d = S.pab[b][p >= sp ? 1 : 0];
            uint32_t *dst = (d & 1ull) ? reinterpret_cast<uint32_t *>(s_xpg[(uint32_t)(d >> 1) + ((p - sp) >> 9)]) + ((p - sp) & (PG_B - 1))
                                       : reinterpret_cast<uint32_t *>(d) + p;
            *dst = v & 0x00FFFFFFu;
        }
        __syncthreads();
    }
    if (tid < NB) { st.page[tid] = my_pg; st.fill[tid] = my_fill; }
    if (tid == 0) st.key = s_cur_key;
}

__global__ void k_pg_close2(ScState *__restrict__ state, const uint8_t *__restrict__ bin_d2,
                            unsigned long long *__restrict__ meta_b, uint32_t *__restrict__ bpcnt,
                            uint32_t *__restrict__ brecs, uint32_t G) {
    const unsigned tid = threadIdx.x;
    ScState &st = state[blockIdx.x];
    const uint32_t key = st.key;
    __syncthreads();                       // everybody has the stream key before thread 0 resets it
    if (tid < 256) {
        const uint32_t pg = st.page[tid], fill = st.fill[tid];
        if (pg != PG_NONE && fill)
            pgb_close(meta_b, bpcnt, brecs, G, pg, ((uint32_t)bin_d2[key & 511u] << 8) | tid, key >> 9, fill);
    }
    if (tid < SC_BINS1) { st.page[tid] = PG_NONE; st.fill[tid] = 0; st.spare[tid] = PG_NONE; }
    if (tid == 0) st.key = 0;
}

// ---- level-2 pages -> bucket page lists ---------------------------------------------------------------
// Pages are listed per (bucket, sample group): key = bucket * G + group, so a bucket's pages are contiguous
// and ordered by group. bpcnt[key] (pages) and brecs[bucket] (records) were counted as k_scatter2 closed the pages.
// The slots a build can have written are those of the level-1 pages of its tiles (their metas were cleared as they
// joined a supply) and the reserve slots it took; every other slot may hold the meta of an earlier build.
__global__ void k_pgb_fill(const unsigned long long *__restrict__ meta, const Sc2Tile *__restrict__ tiles,
                           const uint32_t *__restrict__ ntiles_dev, const uint32_t *__restrict__ cursor_b, uint32_t res0,
                           uint32_t nres, uint32_t G, const unsigned long long *__restrict__ bpstart,
                           uint32_t *__restrict__ bpfill, unsigned long long *__restrict__ blist) {
    const uint64_t ntv = (uint64_t)*ntiles_dev * (2 * SC_TILE_PAGES);
    const uint64_t nv = ntv + min(*cursor_b, nres);
    for (uint64_t v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
        uint32_t slot;
        if (v < ntv) {
            const Sc2Tile &tl = tiles[v / (2 * SC_TILE_PAGES)];
            const uint32_t j = (uint32_t)(v >> 1) % SC_TILE_PAGES;
            if (j >= tl.np) continue;
            slot = 2 * tl.page[j] + (uint32_t)(v & 1);
        } else slot = res0 + (uint32_t)(v - ntv);
        const unsigned long long m = meta[slot];
        if (!m) continue;
        const uint32_t bucket = (uint32_t)(m >> 40), grp = (uint32_t)(m >> 32) & 255u;
        const uint32_t key = bucket * G + grp;
        blist[bpstart[key] + atomicAdd(&bpfill[key], 1u)] = BKP_ENTRY(slot, grp, (uint32_t)m);
    }
}
