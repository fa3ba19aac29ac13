// ps_api.cu — extern "C" entry points of libpskmer.so (see include/pskmer.h) and the host-side
// orchestration of the kernels: ingest/decode -> extract -> radix sort -> rows -> test.
#include <algorithm>
#include <cmath>
#include <numeric>
#include <time.h>

#include "ps_common.cuh"
#include "ps_decode.cuh"
#include "ps_extract.cuh"
#include "ps_sort.cuh"
#include "ps_rows.cuh"
#include "ps_test.cuh"
#include "ps_chi2_reach.h"
#include "ps_mash.cuh"
#include "ps_count.cuh"

static std::string g_create_err;

// PSKMER_TRACE=1: host wall-clock of every API call on stderr (where the host leaves the GPU idle)
struct ApiTrace {
    const char *fn;
    bool on;
    static double now() {
        timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
    }
    ApiTrace(const ps_ctx *c, const char *f) : fn(f), on(c && c->trace_ref) {
        if (on) fprintf(stderr, "[pskmer api] %12.3f enter %s\n", now(), fn);
    }
    ~ApiTrace() {
        if (on) fprintf(stderr, "[pskmer api] %12.3f exit  %s\n", now(), fn);
    }
};

#define API_BEGIN(ctx)                                  \
    if (!(ctx)) return PS_ERR_ARG;                      \
    ApiTrace _api_trace(ctx, __func__);                 \
    try {                                               \
        CK(cudaSetDevice((ctx)->device));

#define API_END(ctx)                                    \
    }                                                   \
    catch (const PsError &e) {                          \
        (ctx)->err = e.msg;                             \
        return e.code;                                  \
    }                                                   \
    catch (const std::exception &e) {                   \
        (ctx)->err = e.what();                          \
        return PS_ERR_NOMEM;                            \
    }                                                   \
    return PS_OK;

static inline bool key64(const ps_ctx *c) { return c->k > 16; }

// ---------------------------------------------------------------------------------------
// digit width: 9 bits when that saves a whole pass over 8-bit digits (k = 13, 17, 18, 21, 22, ...)
static int radix_bits(int bits) { return ((bits + 8) / 9 < (bits + 7) / 8) ? 9 : 8; }
static int radix_passes(int bits, size_t key_bytes, int shift0) {
    const int rb = radix_bits(bits);
    return std::min<int>((bits + rb - 1) / rb, ((int)key_bytes * 8 - shift0 + rb - 1) / rb);
}

// zeroed histogram block of the sort (all passes + the tile counter)
static unsigned long long *radix_hist_reset(ps_ctx *c) {
    c->hist.reserve((size_t)RS_MAX_PASSES * RS_MAX_RADIX * 8 + 64, c->stream);
    CK(cudaMemsetAsync(c->hist.p, 0, (size_t)RS_MAX_PASSES * RS_MAX_RADIX * 8 + 64, c->stream));
    return c->hist.as<unsigned long long>();
}

// radix sort driver: sorts n keys (+ optional u16 tags) by bits [shift0, shift0 + bits); returns
// true if the result is in the *_b buffers.
template <typename KeyT>
static bool radix_sort(ps_ctx *c, KeyT *ka, KeyT *kb, uint16_t *ta, uint16_t *tb, uint64_t n, int bits,
                       bool has_val, int shift0 = 0, bool have_hist = false, double alg_rec_bytes = 0.0) {
    if (n == 0) return false;
    const int npass = radix_passes(bits, sizeof(KeyT), shift0);
    const int rb = radix_bits(bits), radix = 1 << rb;
    const uint64_t tiles = ceil_div<uint64_t>(n, RS_TILE);
    c->lookback.reserve(tiles * radix * 8, c->stream);
    unsigned long long *hist = have_hist ? c->hist.as<unsigned long long>() : radix_hist_reset(c);
    uint32_t *counter = reinterpret_cast<uint32_t *>(hist + RS_MAX_PASSES * RS_MAX_RADIX);
    if (!have_hist) {
        const int hb = (int)std::min<uint64_t>(PS_SMS * 4, ceil_div<uint64_t>(n, 512 * 8));
        KLAUNCH(c, "rs_hist", (double)n * sizeof(KeyT),
                (k_rs_hist<KeyT><<<hb, 512, 0, c->stream>>>(ka, n, npass, shift0, rb, hist)));
    }
    KLAUNCH(c, "rs_scan", 0.0, (k_rs_scan<<<npass, RS_MAX_RADIX, 0, c->stream>>>(hist)));
    bool in_b = false;
    // algorithmic bytes of one record: what a pass must read and write once (for packed records the
    // information content, 2k bits of k-mer + 16 bits of sample tag, not the 8-byte container)
    const double pair_bytes = alg_rec_bytes > 0 ? alg_rec_bytes : (double)(sizeof(KeyT) + (has_val ? 2 : 0));
    for (int p = 0; p < npass; p++) {
        CK(cudaMemsetAsync(c->lookback.p, 0, tiles * radix * 8, c->stream));
        CK(cudaMemsetAsync(counter, 0, 4, c->stream));
        const KeyT *kin = in_b ? kb : ka;
        KeyT *kout = in_b ? ka : kb;
        const uint16_t *vin = in_b ? tb : ta;
        uint16_t *vout = in_b ? ta : tb;
        const int shift = shift0 + rb * p;
        const unsigned long long *gb = hist + (size_t)p * RS_MAX_RADIX;
        unsigned long long *lbk = c->lookback.as<unsigned long long>();
        const char *nm = has_val ? "rs_pass_kv" : "rs_pass_k";
        const unsigned g = (unsigned)tiles;
        if (has_val && rb == 8)
            KLAUNCH(c, nm, 2.0 * n * pair_bytes, (k_rs_pass<KeyT, true, 8><<<g, RS_THREADS, rs_dyn_smem<KeyT, true>(), c->stream>>>(kin, kout, vin, vout, n, shift, gb, lbk, counter)));
        else if (has_val)
            KLAUNCH(c, nm, 2.0 * n * pair_bytes, (k_rs_pass<KeyT, true, 9><<<g, RS_THREADS, rs_dyn_smem<KeyT, true>(), c->stream>>>(kin, kout, vin, vout, n, shift, gb, lbk, counter)));
        else if (rb == 8)
            KLAUNCH(c, nm, 2.0 * n * pair_bytes, (k_rs_pass<KeyT, false, 8><<<g, RS_THREADS, rs_dyn_smem<KeyT, false>(), c->stream>>>(kin, kout, nullptr, nullptr, n, shift, gb, lbk, counter)));
        else
            KLAUNCH(c, nm, 2.0 * n * pair_bytes, (k_rs_pass<KeyT, false, 9><<<g, RS_THREADS, rs_dyn_smem<KeyT, false>(), c->stream>>>(kin, kout, nullptr, nullptr, n, shift, gb, lbk, counter)));
        in_b = !in_b;
    }
    return in_b;
}

// exclusive scan of u32 counts -> u64 offsets (offs[n] = total), on the device
static void scan_counts_dev(ps_ctx *c, const char *name, const uint32_t *counts, uint64_t n, unsigned long long *offs) {
    const uint64_t chunks = std::max<uint64_t>(1, ceil_div<uint64_t>(n, SCAN_CHUNK));
    c->scan_sums.reserve(chunks * 8, c->stream);
    unsigned long long *sums = c->scan_sums.as<unsigned long long>();
    KLAUNCH(c, name, (double)n * 4, (k_scan_sums<<<(unsigned)chunks, SCAN_THREADS, 0, c->stream>>>(counts, n, sums)));
    KLAUNCH(c, name, (double)n * 12, (k_scan_chunks<<<(unsigned)chunks, SCAN_THREADS, 0, c->stream>>>(counts, n, sums, offs)));
}

// exclusive scan of u32 counts -> u64 offsets; returns total (syncs the stream)
static uint64_t scan_counts(ps_ctx *c, const uint32_t *counts, uint64_t n, DevBuf &offs) {
    offs.reserve((n + 1) * 8, c->stream);
    scan_counts_dev(c, "scan_counts", counts, n, offs.as<unsigned long long>());
    return ps_read_scalar<unsigned long long>(c, offs.as<unsigned long long>() + n);
}

// ---------------------------------------------------------------------------------------
// per-sample counting: sorted distinct k-mers of sample idx with count >= cutoff.
// Result left in c->tmp1 (KeyT keys) and c->tmp3 (u32 counts); returns the number kept.
template <typename KeyT>
static uint64_t count_sample(ps_ctx *c, int idx, uint32_t cutoff) {
    c->pre_valid = false;   // uses the sort buffers and histograms
    const SampleInfo &s = c->samples[idx];
    const uint64_t nblocks = s.n_pos / EXT_BLOCK_POS;
    if (nblocks == 0) return 0;
    c->blk_counts.reserve(nblocks * 4, c->stream);
    const uint32_t *seq = c->pool_seq.as<uint32_t>(), *bad = c->pool_bad.as<uint32_t>();
    KLAUNCH(c, "extract_count", (double)s.n_pos * 3 / 8,
            (k_extract<KeyT, false, 0><<<(unsigned)nblocks, EXT_THREADS, 0, c->stream>>>(
                seq, bad, s.pos_off, c->k, 0, 0, 1, nullptr, c->blk_counts.as<uint32_t>(), nullptr,
                nullptr, nullptr)));
    const uint64_t n = scan_counts(c, c->blk_counts.as<uint32_t>(), nblocks, c->blk_offs);
    if (n == 0) return 0;
    c->keys_a.reserve(n * sizeof(KeyT), c->stream);
    c->keys_b.reserve(n * sizeof(KeyT), c->stream);
    KLAUNCH(c, "extract_write", (double)s.n_pos * 3 / 8 + (double)n * sizeof(KeyT),
            (k_extract<KeyT, true, 0><<<(unsigned)nblocks, EXT_THREADS, 0, c->stream>>>(
                seq, bad, s.pos_off, c->k, 0, 0, 1, nullptr, nullptr,
                (const uint64_t *)c->blk_offs.as<unsigned long long>(), c->keys_a.as<KeyT>(), nullptr)));
    const bool in_b = radix_sort<KeyT>(c, c->keys_a.as<KeyT>(), c->keys_b.as<KeyT>(), nullptr, nullptr, n,
                                       2 * c->k, false);
    const KeyT *sorted = in_b ? c->keys_b.as<KeyT>() : c->keys_a.as<KeyT>();
    KeyT *other = in_b ? c->keys_a.as<KeyT>() : c->keys_b.as<KeyT>();
    const uint64_t chunks = ceil_div<uint64_t>(n, RUN_CHUNK);
    const unsigned rb = (unsigned)ceil_div<uint64_t>(chunks, RUN_THREADS / 32);
    c->blk_counts.reserve(chunks * 4, c->stream);
    KLAUNCH(c, "run_count", (double)n * sizeof(KeyT),
            (k_run_count<KeyT><<<rb, RUN_THREADS, 0, c->stream>>>(sorted, n, 0, c->blk_counts.as<uint32_t>())));
    const uint64_t nu = scan_counts(c, c->blk_counts.as<uint32_t>(), chunks, c->blk_offs);
    c->tmp2.reserve(nu * 8, c->stream);
    c->tmp3.reserve(nu * 4, c->stream);
    // distinct keys into `other` (the spare sort buffer), head positions into tmp2
    KLAUNCH(c, "rle_write", (double)n * sizeof(KeyT) + (double)nu * (sizeof(KeyT) + 8),
            (k_rle_write<KeyT><<<rb, RUN_THREADS, 0, c->stream>>>(
                sorted, n, c->blk_offs.as<unsigned long long>(), other, c->tmp2.as<unsigned long long>())));
    const uint64_t uchunks = ceil_div<uint64_t>(nu, RUN_CHUNK);
    const unsigned ub = (unsigned)ceil_div<uint64_t>(uchunks, RUN_THREADS / 32);
    c->blk_counts.reserve(uchunks * 4, c->stream);
    KLAUNCH(c, "rle_counts", (double)nu * 12,
            (k_rle_counts<<<ub, RUN_THREADS, 0, c->stream>>>(c->tmp2.as<unsigned long long>(), nu, n, cutoff,
                                                             c->tmp3.as<uint32_t>(),
                                                             c->blk_counts.as<uint32_t>())));
    const uint64_t kept = scan_counts(c, c->blk_counts.as<uint32_t>(), uchunks, c->blk_offs);
    c->tmp1.reserve(std::max<uint64_t>(kept, 1) * sizeof(KeyT), c->stream);
    // filtered counts reuse tmp2 (head positions are no longer needed after rle_counts)
    uint32_t *out_counts = reinterpret_cast<uint32_t *>(c->tmp2.p);
    KLAUNCH(c, "rle_filter", (double)nu * (sizeof(KeyT) + 4) + (double)kept * (sizeof(KeyT) + 4),
            (k_rle_filter<KeyT><<<ub, RUN_THREADS, 0, c->stream>>>(
                other, c->tmp3.as<uint32_t>(), nu, cutoff, c->blk_offs.as<unsigned long long>(),
                c->tmp1.as<KeyT>(), out_counts)));
    // move the kept counts to tmp3 (device -> device)
    if (kept) CK(cudaMemcpyAsync(c->tmp3.p, out_counts, kept * 4, cudaMemcpyDeviceToDevice, c->stream));
    return kept;
}

// append the counted list in tmp1 to the list pool (list mode)
template <typename KeyT>
static void list_append(ps_ctx *c, int idx, uint64_t kept) {
    SampleInfo &s = c->samples[idx];
    const uint64_t padded = round_up<uint64_t>(std::max<uint64_t>(kept, 1), EXT_BLOCK_POS);
    const uint64_t used_bytes = c->list_used * sizeof(KeyT);
    c->list_keys.reserve((c->list_used + padded) * sizeof(KeyT), c->stream, true, used_bytes);
    if (kept)
        CK(cudaMemcpyAsync(c->list_keys.as<KeyT>() + c->list_used, c->tmp1.p, kept * sizeof(KeyT),
                           cudaMemcpyDeviceToDevice, c->stream));
    s.list_mode = true;
    s.list_off = c->list_used;
    s.list_n = kept;
    c->list_used += padded;
}

// device tables of the bucketed build, carved out of c->blk_offs
struct BucketTables {
    unsigned long long *bstart, *first_row;   // [BK_N + 1] each
    uint32_t *counts, *order, *order2, *fill, *seg_tile0;   // fill[4]
};
static BucketTables bucket_tables(ps_ctx *c) {
    const size_t G = (size_t)std::max(1, (c->n_samples + 255) / 256);      // bstart: one entry per (bucket, sample group)
    c->blk_offs.reserve(((size_t)BK_N * G + 1 + BK_N + 1) * 8 + (size_t)BK_N * 12 + 16 + 257 * 4 + 64, c->stream);
    BucketTables t;
    t.bstart = c->blk_offs.as<unsigned long long>();
    t.first_row = t.bstart + (size_t)BK_N * G + 1;
    t.counts = reinterpret_cast<uint32_t *>(t.first_row + BK_N + 1);
    t.order = t.counts + BK_N;
    t.order2 = t.order + BK_N;
    t.fill = t.order2 + BK_N;
    t.seg_tile0 = t.fill + 4;
    return t;
}

// ---------------------------------------------------------------------------------------
// Paged build (ps_paged.cuh) for k = 9..16: k_scatter1 (extraction fused with the level-1 partition)
// -> page lists -> k_scatter2 -> bucket page lists -> k_bucket_count_pg / k_bucket_build_pg.
static inline bool paged_ok(const ps_ctx *c) { return c->bucketed && c->k >= 9 && c->k <= 16; }
static inline int paged_groups(const ps_ctx *c) { return (c->n_samples + 255) / 256; }

// u32 tables of the paged build inside c->pg_tabs
struct PagedTabs {
    uint32_t *cursor_a;      // [PART_MAX]
    uint32_t *cursor_b, *overflow, *ticket, *ntiles_dummy;
    uint32_t *scnt, *tstart, *sfill;               // [ns], [ns + 1], [ns]
    uint32_t *bpcnt, *brecs, *bpfill;              // [BK_N * G], [BK_N], [BK_N * G]
    uint8_t *bin_d2;                               // [512]
    uint32_t *trash;                               // SC_TILE
    uint32_t ns;
    size_t zero_bytes;                             // prefix that is cleared at the start of every build
};
static PagedTabs paged_tabs(ps_ctx *c) {
    PagedTabs t;
    t.ns = (uint32_t)paged_groups(c) * 512u;
    const size_t G = (size_t)paged_groups(c);
    const size_t words = 16 + (size_t)t.ns * 4 + 2 + (size_t)BK_N * (2 * G + 1) + 128 + SC_TILE + 64;
    c->pg_tabs.reserve(words * 4, c->stream);
    uint32_t *p = c->pg_tabs.as<uint32_t>();
    t.cursor_a = p; t.cursor_b = p + 8; t.overflow = p + 9; t.ticket = p + 10; t.ntiles_dummy = p + 11;
    p += 16;
    t.scnt = p; p += t.ns;
    t.sfill = p; p += t.ns;
    t.bpcnt = p; p += BK_N * G;
    t.brecs = p; p += BK_N;
    t.bpfill = p; p += BK_N * G;
    t.zero_bytes = (size_t)(p - c->pg_tabs.as<uint32_t>()) * 4;
    t.tstart = p; p += t.ns + 1;
    t.bin_d2 = reinterpret_cast<uint8_t *>(p); p += 128;
    t.trash = p;
    return t;
}

// writer's view of this GPU's own level-1 pool (one destination, no splitters)
static Sc1Dst paged_local_dst(ps_ctx *c) {
    const PagedTabs t = paged_tabs(c);
    Sc1Dst d;
    memset(&d, 0, sizeof(d));
    d.nparts = 1;
    d.pool[0].recs = c->keys_a.as<uint32_t>();
    d.pool[0].meta = c->pg_meta_a.as<uint32_t>();
    d.pool[0].page0 = 0;
    d.pool[0].cap = c->pgA_cap;
    d.cursor = t.cursor_a;
    d.overflow = t.overflow;
    d.trash = t.trash;
    return d;
}

// Level-2 reserve (2 KB pages behind the level-1 pages): what k_scatter2's blocks may need beyond the halves of the
// level-1 pages they have read, (streams + 2 x blocks) x 256 pages (the bound is derived in ps_paged.cuh).
static uint64_t paged_reserve_pages(const ps_ctx *c) {
    return ((uint64_t)paged_groups(c) * SC_BINS1 + 2 * c->sc2_grid) * 256 * c->pgR_mult;
}

// The level-1 buffer: cap pages of 4 KB and the level-2 reserve behind them, reserved exactly (it is most of the
// device memory a large job takes). Level-2 slot numbers must fit 32 bits.
static void paged_reserve_pool(ps_ctx *c, uint64_t cap, bool keep) {
    if (keep) cap = std::max<uint64_t>(cap, c->pgA_cap);
    const uint64_t res = paged_reserve_pages(c);
    if (2 * cap + res >= (1ull << 32)) PS_THROW(PS_ERR_NOMEM, "level-1 page pool of %llu pages: cut the job into k-mer ranges", (unsigned long long)cap);
    const uint32_t old_cap = c->pgA_cap;
    c->keys_a.reserve(cap * PG_A * 4 + res * PG_B * 4, c->stream, keep, (size_t)old_cap * PG_A * 4, true);
    c->pg_meta_a.reserve(cap * 4, c->stream, keep, (size_t)old_cap * 4);
    if (keep && cap > old_cap) CK(cudaMemsetAsync(c->pg_meta_a.as<uint32_t>() + old_cap, 0, (cap - old_cap) * 4, c->stream));
    c->pgA_cap = (uint32_t)cap;
    c->pgR_cap = (uint32_t)res;
}

// Level-1 pool for up to n_upper records on this GPU alone (one destination, no splitters). Clears the
// page metas, cursors and block states. keep: the pool already holds live pages (ingest of a later batch).
static Sc1Dst paged_begin_local(ps_ctx *c, uint64_t n_upper, bool keep, uint32_t slack_mult = 1) {
    const PagedTabs t = paged_tabs(c);
    const uint64_t slack = (uint64_t)c->sc1_grid * SC_BINS1 * (paged_groups(c) + 2) * slack_mult;   // open + spare pages
    const uint64_t cap = ceil_div<uint64_t>(n_upper, PG_A) + slack;
    if (!keep || cap > c->pgA_cap || paged_reserve_pages(c) != c->pgR_cap) paged_reserve_pool(c, cap, keep);
    c->pg_state.reserve((size_t)(c->sc1_grid + c->sc2_grid) * sizeof(ScState), c->stream, keep,
                        (size_t)(c->sc1_grid + c->sc2_grid) * sizeof(ScState));
    c->l1_live = false;
    if (!keep) {
        CK(cudaMemsetAsync(c->pg_meta_a.p, 0, (size_t)c->pgA_cap * 4, c->stream));
        CK(cudaMemsetAsync(c->pg_tabs.p, 0, t.zero_bytes, c->stream));
        KLAUNCH(c, "pg_close", 0.0, (k_pg_reset_state<<<c->sc1_grid + c->sc2_grid, 288, 0, c->stream>>>(c->pg_state.as<ScState>())));
    }
    return paged_local_dst(c);
}

static Sc1Src sc1_stream_src(ps_ctx *c, uint64_t pos_begin, uint64_t nblocks, const uint16_t *d_blk_sample) {
    Sc1Src s;
    memset(&s, 0, sizeof(s));
    s.seq = c->pool_seq.as<uint32_t>();
    s.bad = c->pool_bad.as<uint32_t>();
    s.blk_sample = d_blk_sample;
    s.pos_begin = pos_begin;
    s.nblocks = nblocks;
    s.k = c->k;
    s.lo = c->range_all ? 0u : (uint32_t)c->range_lo;
    const uint64_t space = 1ull << (2 * c->k);
    s.hi = (c->range_all || c->range_hi >= space) ? 0xFFFFFFFFu : (uint32_t)(c->range_hi - 1);
    return s;
}

template <int SRC>
static void launch_scatter1(ps_ctx *c, const Sc1Src &src, const Sc1Dst &dst) {
    if (src.nblocks == 0) return;
    const PagedTabs t = paged_tabs(c);
    CK(cudaMemsetAsync(t.ticket, 0, 4, c->stream));
    const uint32_t tiles = (uint32_t)((src.nblocks + 1) / 2);
    const int grid = (int)std::min<uint32_t>((uint32_t)c->sc1_grid, tiles);
    const size_t smem = (size_t)SC_TILE * 6 + sizeof(ScShared<SC_BINS1>);
    const double pos = (double)src.nblocks * EXT_BLOCK_POS;
    // The recomputing variant (3 blocks per SM) wins on one GPU and whenever a range filter drops part of the
    // k-mers; with peer pools in the write-out and every k-mer kept, the register variant (2 blocks per SM) is faster
    // (measured at 2 GPUs: config 3 17.6 vs 23.2 ms, config 2 3.81 vs 3.96 ms; config 5 in two passes: 117 vs 105 ms).
    const bool all_kept = src.lo == 0u && src.hi == 0xFFFFFFFFu;
    if (SRC == 0 && c->sc1_lean && (dst.nparts <= 1 || !all_kept))
        KLAUNCH(c, "scatter1", pos * (3.0 / 8 + 4 * c->sc1_out_frac),
                (k_scatter1<0, true><<<grid, SC_THREADS, smem, c->stream>>>(src, dst, c->pg_state.as<ScState>(), t.ticket)));
    else
        KLAUNCH(c, "scatter1", SRC == 0 ? pos * (3.0 / 8 + 4 * c->sc1_out_frac) : pos * (4 + 4 * c->sc1_out_frac),
                (k_scatter1<SRC, false><<<std::min(grid, 2 * PS_SMS), SC_THREADS, smem, c->stream>>>(src, dst, c->pg_state.as<ScState>(), t.ticket)));
}

// Thrown by paged_finish when records did not fit the page pools (PS_ERR_NOMEM): callers that can take larger pools
// catch this type and build again (a larger reserve if the level-2 reserve ran out: pgR_mult has doubled). k_scatter2
// has then written over level-1 pages of the build's bins: the records must be extracted again.
struct PagePoolExhausted : PsError {};

// ps_scatter_range's pool: which level-1 bins a build has consumed
static bool l1_consumed(const ps_ctx *c, uint32_t blo, uint32_t bhi) {
    for (uint32_t b = blo; b < bhi; b++)
        if ((c->l1_used[b >> 6] >> (b & 63)) & 1ull) return true;
    return false;
}
static void l1_consume(ps_ctx *c, uint32_t blo, uint32_t bhi) {
    for (uint32_t b = blo; b < bhi; b++) c->l1_used[b >> 6] |= 1ull << (b & 63);
}

// level-1 pages (this GPU's pool, pgA_cap pages, metas final) -> union + matrix
// bin_lo / bin_hi: only the level-1 bins [bin_lo, bin_hi) take part (a sub-range of what the pool was scattered
// for); rezero: the tables of an earlier paged_finish on the same pool are cleared first (everything but the
// level-1 page cursors).
static void paged_finish(ps_ctx *c, const Sc1Dst &dst_for_close, bool close_local, const uint8_t *h_bin_d2, uint64_t n_upper,
                         uint32_t bin_lo = 0, uint32_t bin_hi = 512, bool rezero = false) {
    const PagedTabs t = paged_tabs(c);
    const int lbits = 2 * c->k - 16;
    ScState *st1 = c->pg_state.as<ScState>(), *st2 = st1 + c->sc1_grid;
    if (rezero) CK(cudaMemsetAsync(t.cursor_b, 0, t.zero_bytes - 8 * 4, c->stream));
    if (close_local)
        KLAUNCH(c, "pg_close", 0.0, (k_pg_close1<<<c->sc1_grid, 288, 0, c->stream>>>(st1, dst_for_close, lbits)));
    CK(cudaMemcpyAsync(t.bin_d2, h_bin_d2, 512, cudaMemcpyHostToDevice, c->stream));
    const uint32_t npa = c->pgA_cap;
    c->pg_tiles.reserve(((size_t)npa / SC_TILE_PAGES + t.ns + 1) * sizeof(Sc2Tile), c->stream);
    KLAUNCH(c, "pga_hist", (double)npa * 4,
            (k_pga_pages<false><<<ceil_div<uint32_t>(npa, PGL_THREADS * PGL_PER), PGL_THREADS, 0, c->stream>>>(
                c->pg_meta_a.as<uint32_t>(), npa, bin_lo, bin_hi, t.scnt, t.tstart, t.sfill, c->pg_tiles.as<Sc2Tile>())));
    KLAUNCH(c, "pga_scan", (double)t.ns * 12, (k_pga_scan<<<1, 1024, 0, c->stream>>>(t.scnt, t.ns, t.tstart, t.sfill)));
    KLAUNCH(c, "pga_fill", (double)npa * 4,
            (k_pga_pages<true><<<ceil_div<uint32_t>(npa, PGL_THREADS * PGL_PER), PGL_THREADS, 0, c->stream>>>(
                c->pg_meta_a.as<uint32_t>(), npa, bin_lo, bin_hi, t.scnt, t.tstart, t.sfill, c->pg_tiles.as<Sc2Tile>())));
    // level 2 writes its pages into the halves of the level-1 pages it has read, then into the reserve behind them
    const uint64_t nslots = 2ull * npa + c->pgR_cap;
    c->pg_meta_b.reserve(nslots * 8, c->stream);
    const uint32_t G = (uint32_t)paged_groups(c);
    Sc2Args a;
    a.recs = c->keys_a.as<uint32_t>();
    a.tiles = c->pg_tiles.as<Sc2Tile>();
    a.ntiles = t.tstart + t.ns; a.bin_d2 = t.bin_d2;
    a.meta_b = c->pg_meta_b.as<unsigned long long>();
    a.res0 = 2 * npa; a.nres = c->pgR_cap; a.cursor_b = t.cursor_b; a.overflow = t.overflow; a.trash = t.trash;
    a.bpcnt = t.bpcnt; a.brecs = t.brecs; a.G = G;
    KLAUNCH(c, "scatter2", (double)n_upper * 8, (k_scatter2<<<c->sc2_grid, SC_THREADS, SC2_SMEM, c->stream>>>(a, st2)));
    KLAUNCH(c, "pg_close", 0.0, (k_pg_close2<<<c->sc2_grid, 288, 0, c->stream>>>(st2, t.bin_d2, a.meta_b, t.bpcnt, t.brecs, G)));
    // bucket page lists
    const BucketTables bt = bucket_tables(c);
    CK(cudaMemsetAsync(bt.fill, 0, 16, c->stream));
    const int lg = PS_SMS * 8;
    scan_counts_dev(c, "scan_bpages", t.bpcnt, (uint64_t)BK_N * G, bt.bstart);
    c->pg_blist.reserve((size_t)nslots * 8, c->stream);
    KLAUNCH(c, "pgb_fill", (double)npa * 20, (k_pgb_fill<<<lg, 256, 0, c->stream>>>(a.meta_b, a.tiles, a.ntiles, t.cursor_b, a.res0, a.nres, G,
                                                                                 bt.bstart, t.bpfill, c->pg_blist.as<unsigned long long>())));
    KLAUNCH(c, "bucket_order", (double)BK_N * 8, (k_bucket_order_pg<<<BK_N / 256, 256, 0, c->stream>>>(
                                     t.brecs, (uint32_t)std::min<uint64_t>(4 * (n_upper / BK_N) + 4096, 0xFFFFFFFFu), bt.fill, bt.order)));
    const int nwords = lbits >= 5 ? (1 << (lbits - 5)) : 1;
    c->tmp1.reserve((size_t)BK_N * nwords * 4, c->stream);
    uint32_t *gbm = c->tmp1.as<uint32_t>();
    KLAUNCH(c, "bucket_count", (double)n_upper * 4,
            (k_bucket_count_pg<<<BK_N, BK_THREADS, 0, c->stream>>>(
                a.recs, c->pg_blist.as<unsigned long long>(), bt.bstart, G, bt.order, lbits, bt.counts, gbm)));
    scan_counts_dev(c, "scan_rows", bt.counts, BK_N, bt.first_row);
    const uint32_t stride = (uint32_t)std::min(c->row_words, 8) + 1;      // rows are assembled in 8-word column slices
    const uint32_t cap_small = (uint32_t)std::max(c->bk_row_words, round_up<int>((int)stride, 4));
    const uint32_t cap_big = (uint32_t)std::max<int>((BK_MAX_DYN_SMEM - nwords * 8) / 4 & ~3, (int)cap_small);
    KLAUNCH(c, "bucket_order", (double)BK_N * 8,
            (k_bucket_order_pg<<<BK_N / 256, 256, 0, c->stream>>>(bt.counts, cap_small / stride, bt.fill + 2, bt.order2)));
    unsigned long long *h = (unsigned long long *)ps_pinned(c, 64);
    uint32_t *h32 = reinterpret_cast<uint32_t *>(h + 1);
    CK(cudaMemcpyAsync(h, bt.first_row + BK_N, 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h32, bt.fill + 2, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h32 + 1, t.overflow, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h32 + 2, t.cursor_a, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h32 + 3, t.cursor_b, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (h32[1]) {
        char m[160];
        snprintf(m, sizeof(m), "page pool exhausted (level-1 %u of %u pages, level-2 reserve %u of %u)", h32[2], c->pgA_cap, h32[3], c->pgR_cap);
        if (h32[3] > c->pgR_cap) c->pgR_mult *= 2;
        throw PagePoolExhausted{{PS_ERR_NOMEM, m}};
    }
    const uint64_t U = h[0];
    const uint32_t nbig = h32[0];
    c->U = U;
    const size_t row_bytes = (size_t)c->row_words * 4;
    c->uni.reserve(std::max<uint64_t>(U, 1) * 8, c->stream);
    c->matrix.reserve(U * row_bytes + 64, c->stream);
    const double alg = (double)n_upper * 4 + (double)U * (8 + row_bytes);
    const size_t sm_small = (size_t)cap_small * 4 + (size_t)nwords * 8;
    const size_t sm_big = (size_t)cap_big * 4 + (size_t)nwords * 8;
    const unsigned long long *blist = c->pg_blist.as<unsigned long long>();
    if (nbig)
        KLAUNCH(c, "bucket_build", alg * nbig / BK_N,
                (k_bucket_build_pg<BK_MAX_THREADS><<<nbig, BK_MAX_THREADS, sm_big, c->stream>>>(
                    a.recs, blist, bt.bstart, G, bt.order2, bt.first_row, gbm, lbits, c->row_words, cap_big,
                    c->uni.as<uint64_t>(), c->matrix.as<uint32_t>())));
    if (nbig < BK_N)
        KLAUNCH(c, "bucket_build", alg * (BK_N - nbig) / BK_N,
                (k_bucket_build_pg<BK_THREADS><<<BK_N - nbig, BK_THREADS, sm_small, c->stream>>>(
                    a.recs, blist, bt.bstart, G, bt.order2 + nbig, bt.first_row, gbm, lbits, c->row_words, cap_small,
                    c->uni.as<uint64_t>(), c->matrix.as<uint32_t>())));
}

// single-GPU bin -> d2 table (bin = d2, one destination)
static void bin_d2_identity(uint8_t *tab) {
    for (int i = 0; i < 512; i++) tab[i] = (uint8_t)std::min(i, 255);
}

// ---------------------------------------------------------------------------------------
template <typename KeyT>
static void add_samples_impl(ps_ctx *c, int first_idx, int count, const void *const *bytes,
                             const size_t *lens) {
    // 1. stage the raw text on the device. Text that already lives in device memory at a 16-byte
    // aligned address is decoded in place (FileEnt.off is an absolute device address; the decode
    // kernels get a null base): no staging copy, no staging memory.
    bool from_host = true;
    for (int i = 0; i < count; i++)
        if (lens[i]) {
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, bytes[i]) == cudaSuccess)
                from_host = !(at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged);
            else cudaGetLastError();
            break;
        }
    std::vector<uint8_t> in_place(count, 0);
    std::vector<FileEnt> files(count);
    std::vector<uint32_t> tile_file;
    uint64_t off = 0;
    uint32_t tiles = 0;
    for (int i = 0; i < count; i++) {
        if (lens[i] >= (1ull << 32) - 4096) PS_THROW(PS_ERR_ARG, "sample %d: input larger than 4 GiB", first_idx + i);
        FileEnt &f = files[i];
        memset(&f, 0, sizeof(f));
        f.off = off;
        f.len = lens[i];
        f.tile0 = tiles;
        f.ntiles = (uint32_t)std::max<uint64_t>(1, ceil_div<uint64_t>(lens[i], DEC_TILE));
        tiles += f.ntiles;
        in_place[i] = !from_host && lens[i] && (reinterpret_cast<uintptr_t>(bytes[i]) & 15) == 0;
        if (!in_place[i]) off += round_up<uint64_t>(lens[i], 16) + 16;
    }
    tile_file.resize(tiles);
    for (int i = 0; i < count; i++)
        for (uint32_t t = 0; t < files[i].ntiles; t++) tile_file[files[i].tile0 + t] = (uint32_t)i;
    c->staging.reserve(off + 64, c->stream);
    for (int i = 0; i < count; i++)
        files[i].off = in_place[i] ? (uint64_t)reinterpret_cast<uintptr_t>(bytes[i])
                                   : (uint64_t)reinterpret_cast<uintptr_t>(c->staging.as<uint8_t>()) + files[i].off;
    c->file_tab.reserve(count * sizeof(FileEnt), c->stream);
    c->tile_tab.reserve((size_t)tiles * 4 * 3, c->stream);  // tile_file | tile_state | tile_off
    // tile_cnt (u64) | tile_next (u32) | per-chunk summaries of pass 1, reused by pass 2: cnt (u64) | next (u32)
    c->tile_sum.reserve((size_t)tiles * 12 + (size_t)tiles * DEC_THREADS * 12 + 64, c->stream);
    FileEnt *d_files = c->file_tab.as<FileEnt>();
    uint32_t *d_tile_file = c->tile_tab.as<uint32_t>();
    uint32_t *d_tile_state = d_tile_file + tiles, *d_tile_off = d_tile_state + tiles;
    uint64_t *d_tile_cnt = c->tile_sum.as<uint64_t>();
    uint32_t *d_tile_next = reinterpret_cast<uint32_t *>(d_tile_cnt + tiles);
    uint64_t *d_chunk_cnt = d_tile_cnt + tiles + (tiles + 1) / 2;   // 8-byte aligned, behind tile_next
    uint32_t *d_chunk_next = reinterpret_cast<uint32_t *>(d_chunk_cnt + (size_t)tiles * DEC_THREADS);
    const uint8_t *stg = nullptr;   // FileEnt.off is absolute
    // Host text is ingested in groups of ~64 MB: all uploads are queued on the copy stream at
    // once, and group g is decoded on the compute stream while groups g+1.. are still crossing
    // PCIe. Device-resident text is one group (no transfer to hide).
    const uint64_t group_bytes = from_host ? (64ull << 20) : ~0ull;
    std::vector<int> gstart{0};
    {
        uint64_t acc = 0;
        for (int i = 0; i < count; i++) {
            if (acc > 0 && acc + lens[i] > group_bytes) { gstart.push_back(i); acc = 0; }
            acc += lens[i];
        }
        gstart.push_back(count);
    }
    const int ngroups = (int)gstart.size() - 1;
    // worst case one position per input byte: reserve the pool once, it never moves mid-ingest
    const uint64_t pool0 = c->pool_pos;
    {
        uint64_t ub = pool0;
        for (int i = 0; i < count; i++) ub += round_up<uint64_t>(lens[i] + 1, POS_ALIGN);
        c->pool_seq.reserve(ub / 4 + 64, c->stream, true, pool0 / 4);
        c->pool_bad.reserve(ub / 8 + 64, c->stream, true, pool0 / 8);
    }
    CK(cudaMemcpyAsync(d_files, files.data(), count * sizeof(FileEnt), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d_tile_file, tile_file.data(), (size_t)tiles * 4, cudaMemcpyHostToDevice, c->stream));
    // Host input, whole k-mer space, cutoff 1, k <= 24: the packed records of a group are extracted
    // (and the radix histograms accumulated) right after the group is decoded, i.e. while the next
    // groups are still crossing PCIe; ps_build_union then starts with the sort.
    // ps_ingest_scatter: the same for ONE k-mer range of a job that is built in ranges (the range's level-1 pool
    // was sized by the caller; ps_scatter_range for that range then finds its work done)
    const bool ing = c->ing_on && c->cutoff == 1 && paged_ok(c) && c->route_n <= 1 &&
                     (pool0 == 0 || (c->pre_valid && c->pgA_live && c->pre_ranged && c->pre_n == pool0));
    bool pre = ing || (from_host && ngroups > 1 && c->cutoff == 1 && paged_ok(c) && c->range_all && c->route_n <= 1 && !c->ing_on &&
                       (pool0 == 0 || (c->pre_valid && c->pgA_live && !c->pre_ranged && c->pre_n == pool0)));
    uint16_t *d_pre_tab = nullptr;
    std::vector<uint16_t> pre_tab;
    Sc1Dst pre_dst;
    if (pre && !ing) {
        uint64_t ub = pool0;
        for (int i = 0; i < count; i++) ub += round_up<uint64_t>(lens[i] + 1, POS_ALIGN);
        // scattering during ingest only pays when the whole job fits at once (the level-1 page pool, 4 B per
        // instance, within a third of the free memory); larger jobs are built in k-mer ranges later
        size_t mem_free = 0, mem_total = 0;
        cudaMemGetInfo(&mem_free, &mem_total);
        const uint64_t have = (uint64_t)mem_free + c->keys_a.cap + c->keys_b.cap;
        if (ub * 4 > have / 3) pre = false;
    }
    if (pre) {
        uint64_t ub = pool0;
        for (int i = 0; i < count; i++) ub += round_up<uint64_t>(lens[i] + 1, POS_ALIGN);
        pre_dst = paged_begin_local(c, ing ? std::max<uint64_t>(c->ing_n, EXT_BLOCK_POS) : ub, pool0 != 0);
        c->samp_tab.reserve(ub / EXT_BLOCK_POS * 2 + 256, c->stream, true, pool0 / EXT_BLOCK_POS * 2);
        d_pre_tab = c->samp_tab.as<uint16_t>();
        c->pre_valid = true;
        c->pgA_live = true;
        c->pre_ranged = ing;
        c->pre_lo = ing ? c->ing_lo : 0;
        c->pre_hi = ing ? c->ing_hi : 0;
    } else {
        c->pre_valid = false;
        c->pgA_live = false;
    }
    std::vector<cudaEvent_t> ev(ngroups, nullptr);
    if (ngroups > 1) {
        if (!c->copy_stream) CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        cudaEvent_t e0;
        CK(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
        CK(cudaEventRecord(e0, c->stream));              // staging buffer is ready (reserve may have synced)
        CK(cudaStreamWaitEvent(c->copy_stream, e0, 0));
        cudaEventDestroy(e0);
    }
    cudaStream_t cs = ngroups > 1 ? c->copy_stream : c->stream;
    for (int g = 0; g < ngroups; g++) {
        for (int i = gstart[g]; i < gstart[g + 1]; i++)
            if (lens[i] && !in_place[i])
                CK(cudaMemcpyAsync(reinterpret_cast<void *>((uintptr_t)files[i].off), bytes[i], lens[i], cudaMemcpyDefault, cs));
        if (ngroups > 1) {
            CK(cudaEventCreateWithFlags(&ev[g], cudaEventDisableTiming));
            CK(cudaEventRecord(ev[g], cs));
        }
    }
    uint64_t pp = pool0;
    for (int g = 0; g < ngroups; g++) {
        const int f0 = gstart[g], nf = gstart[g + 1] - gstart[g];
        const uint32_t t0 = files[f0].tile0;
        const uint32_t nt = files[f0 + nf - 1].tile0 + files[f0 + nf - 1].ntiles - t0;
        uint64_t gbytes = 0;
        for (int i = f0; i < f0 + nf; i++) gbytes += lens[i];
        if (ngroups > 1) CK(cudaStreamWaitEvent(c->stream, ev[g], 0));
        KLAUNCH(c, "detect", 0.0, (k_detect<<<nf, 256, 0, c->stream>>>(stg, d_files + f0)));
        KLAUNCH(c, "decode_count", (double)gbytes,
                (k_decode_count<<<nt, DEC_THREADS, 0, c->stream>>>(stg, d_files, d_tile_file, t0, d_tile_next,
                                                                   d_tile_cnt, d_chunk_next, d_chunk_cnt)));
        KLAUNCH(c, "decode_walk", (double)nt * 20,
                (k_decode_walk<<<ceil_div(nf, 64), 64, 0, c->stream>>>(d_files + f0, nf, d_tile_next, d_tile_cnt,
                                                                       d_tile_state, d_tile_off)));
        // stream lengths of this group -> pool layout
        CK(cudaMemcpyAsync(files.data() + f0, d_files + f0, nf * sizeof(FileEnt), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        const uint64_t gp0 = pp;
        for (int i = f0; i < f0 + nf; i++) {
            files[i].n_pos = round_up<uint64_t>(files[i].m + 1, POS_ALIGN);
            files[i].pool_off = pp;
            pp += files[i].n_pos;
        }
        CK(cudaMemsetAsync(c->pool_seq.as<uint8_t>() + gp0 / 4, 0, (pp - gp0) / 4, c->stream));
        CK(cudaMemsetAsync(c->pool_bad.as<uint8_t>() + gp0 / 8, 0, (pp - gp0) / 8, c->stream));
        CK(cudaMemcpyAsync(d_files + f0, files.data() + f0, nf * sizeof(FileEnt), cudaMemcpyHostToDevice, c->stream));
        uint32_t fmt_seen = 0;                       // bit f set: some file of the group has format f
        for (int i = f0; i < f0 + nf; i++) fmt_seen |= 1u << files[i].fmt;
        fmt_seen &= ~1u;
        // all FASTA: the word-wide write pass; otherwise the byte transducer, FASTQ-only or per file
        auto *write = fmt_seen == 2u ? k_decode_write_fasta : fmt_seen == 4u ? k_decode_write<2> : k_decode_write<0>;
        KLAUNCH(c, "decode_write", (double)gbytes + (double)(pp - gp0) * 3 / 8,
                (write<<<nt, DEC_THREADS, 0, c->stream>>>(stg, d_files, d_tile_file, t0, d_tile_state, d_tile_off, d_chunk_next,
                                                          d_chunk_cnt, c->pool_seq.as<uint32_t>(), c->pool_bad.as<uint32_t>())));
        for (int i = f0; i < f0 + nf; i++) if (files[i].fmt == 2) pre = false;   // raw reads: counted per sample
        if (!pre) { c->pre_valid = false; c->pgA_live = false; }
        if (pre && pp > gp0) {
            const uint64_t b0 = gp0 / EXT_BLOCK_POS, nb = (pp - gp0) / EXT_BLOCK_POS;
            pre_tab.clear();
            for (int i = f0; i < f0 + nf; i++)
                pre_tab.insert(pre_tab.end(), files[i].n_pos / EXT_BLOCK_POS, (uint16_t)(first_idx + i));
            CK(cudaMemcpyAsync(d_pre_tab + b0, pre_tab.data(), nb * 2, cudaMemcpyHostToDevice, c->stream));
            if (ing) {
                // extraction honours the context's range: the ingest range for this launch only
                const uint64_t keep_lo = c->range_lo, keep_hi = c->range_hi;
                const bool keep_all = c->range_all;
                c->range_lo = c->ing_lo; c->range_hi = c->ing_hi ? c->ing_hi : ~0ull; c->range_all = (c->ing_lo == 0 && c->ing_hi == 0);
                c->sc1_out_frac = c->ing_share;
                const Sc1Src src1 = sc1_stream_src(c, gp0, nb, d_pre_tab);
                c->range_lo = keep_lo; c->range_hi = keep_hi; c->range_all = keep_all;
                launch_scatter1<0>(c, src1, pre_dst);
                c->sc1_out_frac = 1.0;
            } else
                launch_scatter1<0>(c, sc1_stream_src(c, gp0, nb, d_pre_tab), pre_dst);
            CK(cudaStreamSynchronize(c->stream));   // pre_tab is reused by the next group
            c->pre_n = pp;
        }
    }
    for (auto e : ev) if (e) cudaEventDestroy(e);
    CK(cudaStreamSynchronize(c->stream));   // `files` (host vector) was the source of async copies
    c->pool_pos = pp;
    for (int i = 0; i < count; i++) {
        SampleInfo &s = c->samples[first_idx + i];
        s.present = true;
        s.list_mode = false;
        s.pos_off = files[i].pool_off;
        s.n_pos = files[i].n_pos;
    }
    // 3. raw reads, or a cutoff: count per sample now and keep only the counted list
    for (int i = 0; i < count; i++) {
        if (files[i].fmt == 2 || c->cutoff > 1) {
            const uint64_t kept = count_sample<KeyT>(c, first_idx + i, c->cutoff);
            list_append<KeyT>(c, first_idx + i, kept);
        }
    }
    c->have_union = false;
}

// ---------------------------------------------------------------------------------------
// sorted packed records -> union + bit matrix
static void build_rows_packed(ps_ctx *c, const uint64_t *sr, uint64_t n) {
    const uint64_t chunks = ceil_div<uint64_t>(n, RUN_CHUNK);
    const unsigned rb = (unsigned)ceil_div<uint64_t>(chunks, RUN_THREADS / 32);
    c->blk_counts.reserve(chunks * 4, c->stream);
    KLAUNCH(c, "run_count", (double)n * 8,
            (k_run_count<uint64_t><<<rb, RUN_THREADS, 0, c->stream>>>(sr, n, 16, c->blk_counts.as<uint32_t>())));
    const uint64_t U = scan_counts(c, c->blk_counts.as<uint32_t>(), chunks, c->blk_offs);
    c->U = U;
    const size_t mbytes = (size_t)U * c->row_words * 4;
    c->uni.reserve(std::max<uint64_t>(U, 1) * 8, c->stream);
    c->matrix.reserve(mbytes + 64, c->stream);
    CK(cudaMemsetAsync(c->matrix.p, 0, mbytes, c->stream));
    KLAUNCH(c, "row_build", (double)n * 8 + (double)U * 8 + (double)mbytes,
            (k_row_build<uint64_t, true><<<rb, RUN_THREADS, 0, c->stream>>>(
                sr, nullptr, n, c->blk_offs.as<unsigned long long>(), c->uni.as<uint64_t>(),
                c->matrix.as<uint32_t>(), c->row_words)));
}

// full-sort path (k <= 8, k > 16, PSKMER_ROWS=sorted): sort n packed records by k-mer, then run heads -> rows
static void sort_and_build_packed(ps_ctx *c, uint64_t *ra, uint64_t *rb, uint64_t n) {
    const double alg = (2 * c->k + 7) / 8 + 2.0;
    const bool in_b = radix_sort<uint64_t>(c, ra, rb, nullptr, nullptr, n, 2 * c->k, false, 16, false, alg);
    build_rows_packed(c, in_b ? rb : ra, n);
}

// Where the k-mer instances of a job come from: maximal runs of stream-mode samples in the pool
// ("stream segments", positions) and the counted lists of raw-read / cutoff samples ("list segments",
// entries), each cut into blocks of 4096 with the sample of every block in a device table.
struct SegPlan {
    std::vector<Segment> segs;
    uint64_t stream_blocks = 0, nblk = 0;
    bool any_list = false;
    const uint16_t *d_blk_sample = nullptr;    // indexed by absolute pool block
    const uint16_t *d_list_sample = nullptr;   // indexed by list block (nblk - stream_blocks of them)
    const uint32_t *d_list_valid = nullptr;
};
static SegPlan plan_segments(ps_ctx *c, bool require_all) {
    SegPlan P;
    std::vector<std::pair<uint64_t, int>> order;  // (pos_off, idx)
    for (int i = 0; i < c->n_samples; i++) {
        if (!c->samples[i].present) {
            if (require_all) PS_THROW(PS_ERR_STATE, "sample %d was never added", i);
            continue;
        }
        order.push_back({c->samples[i].pos_off, i});
    }
    std::sort(order.begin(), order.end());
    std::vector<uint16_t> blk_sample;   // per extraction block (pool-indexed)
    std::vector<uint32_t> blk_valid;    // list blocks only
    const uint64_t pool_blocks = c->pool_pos / EXT_BLOCK_POS;
    blk_sample.assign(pool_blocks, 0);
    uint64_t nblk = 0;
    for (auto &pr : order) {
        const SampleInfo &s = c->samples[pr.second];
        for (uint64_t b = 0; b < s.n_pos / EXT_BLOCK_POS; b++) blk_sample[s.pos_off / EXT_BLOCK_POS + b] = (uint16_t)pr.second;
        if (s.list_mode) continue;
        if (!P.segs.empty() && !P.segs.back().list &&
            P.segs.back().begin + P.segs.back().nblocks * EXT_BLOCK_POS == s.pos_off)
            P.segs.back().nblocks += s.n_pos / EXT_BLOCK_POS;
        else
            P.segs.push_back({s.pos_off, s.n_pos / EXT_BLOCK_POS, nblk, false});
        nblk += s.n_pos / EXT_BLOCK_POS;
    }
    P.stream_blocks = nblk;
    std::vector<uint16_t> list_blk_sample;
    for (auto &pr : order) {
        const SampleInfo &s = c->samples[pr.second];
        if (!s.list_mode) continue;
        const uint64_t lb = round_up<uint64_t>(std::max<uint64_t>(s.list_n, 1), EXT_BLOCK_POS) / EXT_BLOCK_POS;
        P.segs.push_back({s.list_off, lb, nblk, true});
        for (uint64_t b = 0; b < lb; b++) {
            list_blk_sample.push_back((uint16_t)pr.second);
            const uint64_t done = b * EXT_BLOCK_POS;
            blk_valid.push_back((uint32_t)std::min<uint64_t>(EXT_BLOCK_POS, s.list_n > done ? s.list_n - done : 0));
        }
        nblk += lb;
    }
    P.nblk = nblk;
    P.any_list = !list_blk_sample.empty();
    // device tables: [pool-indexed u16 sample ids][list-block u16 sample ids][list-block valid u32]
    const size_t tab_bytes = round_up<size_t>(pool_blocks * 2, 16) + round_up<size_t>(list_blk_sample.size() * 2, 16) +
                             blk_valid.size() * 4 + 64;
    c->samp_tab.reserve(tab_bytes, c->stream);
    uint16_t *d_blk_sample = c->samp_tab.as<uint16_t>();
    uint16_t *d_list_sample = reinterpret_cast<uint16_t *>(c->samp_tab.as<uint8_t>() + round_up<size_t>(pool_blocks * 2, 16));
    uint32_t *d_list_valid = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(d_list_sample) +
                                                          round_up<size_t>(list_blk_sample.size() * 2, 16));
    if (pool_blocks)
        CK(cudaMemcpyAsync(d_blk_sample, blk_sample.data(), pool_blocks * 2, cudaMemcpyHostToDevice, c->stream));
    if (!list_blk_sample.empty()) {
        CK(cudaMemcpyAsync(d_list_sample, list_blk_sample.data(), list_blk_sample.size() * 2, cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemcpyAsync(d_list_valid, blk_valid.data(), blk_valid.size() * 4, cudaMemcpyHostToDevice, c->stream));
    }
    P.d_blk_sample = d_blk_sample; P.d_list_sample = d_list_sample; P.d_list_valid = d_list_valid;
    return P;
}

// k_scatter1 over every segment of the plan into `d`
static void scatter_segments(ps_ctx *c, const SegPlan &P, const Sc1Dst &d) {
    for (auto &sg : P.segs) {
        if (!sg.list) {
            launch_scatter1<0>(c, sc1_stream_src(c, sg.begin, sg.nblocks, P.d_blk_sample), d);
        } else {
            Sc1Src src = sc1_stream_src(c, sg.begin, sg.nblocks, P.d_list_sample + (sg.blk0 - P.stream_blocks));
            src.list_keys = reinterpret_cast<const uint32_t *>(c->list_keys.p);
            src.blk_valid = P.d_list_valid + (sg.blk0 - P.stream_blocks);
            launch_scatter1<1>(c, src, d);
        }
    }
}

template <typename KeyT>
static void build_union_impl(ps_ctx *c) {
    const SegPlan P = plan_segments(c, true);
    const std::vector<Segment> &segs = P.segs;
    const uint64_t stream_blocks = P.stream_blocks, nblk = P.nblk;
    const uint16_t *d_blk_sample = P.d_blk_sample, *d_list_sample = P.d_list_sample;
    const uint32_t *d_list_valid = P.d_list_valid;
    c->row_words = (int)round_up<int>(ceil_div<int>(c->n_samples, 32), 4);
    if (paged_ok(c)) {
        // k = 9..16: extraction (or the counted lists) -> pages -> buckets -> union + matrix
        c->U = 0; c->have_union = true; c->n_surv = 0;
        const bool have_pre = c->pre_valid && c->pgA_live && !c->pre_ranged && c->range_all && !P.any_list && segs.size() == 1 &&
                              segs[0].begin == 0 && c->pre_n == stream_blocks * EXT_BLOCK_POS;
        c->pre_valid = false;
        c->pgA_live = false;
        if (nblk == 0) return;
        const uint64_t n_all = nblk * EXT_BLOCK_POS;
        uint64_t n_upper = (!c->range_all && c->cap_hint) ? std::min<uint64_t>(c->cap_hint, n_all) : n_all;
        uint8_t bin_d2[512];
        bin_d2_identity(bin_d2);
        if (c->l1_live && c->route_n <= 1) {
            // the range is a run of level-1 bins of the pool ps_scatter_range left: no extraction, only the
            // pages of those bins go through level 2 and the bucket kernels
            const int bshift = 2 * c->k - 8;
            const uint64_t space = 1ull << (2 * c->k);
            const uint64_t lo = c->range_all ? 0 : c->range_lo, hi = (c->range_all || c->range_hi >= space) ? space : c->range_hi;
            const uint64_t l1hi = c->l1_hi == 0 ? space : c->l1_hi;
            const bool lo_ok = lo == c->l1_lo || (lo > c->l1_lo && (lo & ((1ull << bshift) - 1)) == 0);
            const bool hi_ok = hi == l1hi || (hi < l1hi && (hi & ((1ull << bshift) - 1)) == 0);
            const uint32_t blo = (uint32_t)(lo >> bshift), bhi = lo < hi ? (uint32_t)((hi - 1) >> bshift) + 1 : 0u;
            if (lo_ok && hi_ok && lo < hi && !l1_consumed(c, blo, bhi)) {
                // level 2 writes over the level-1 pages of these bins: a later build of them extracts again
                l1_consume(c, blo, bhi);
                try {
                    paged_finish(c, paged_local_dst(c), false, bin_d2, std::min<uint64_t>(n_upper, c->l1_instances), blo, bhi, true);
                    return;
                } catch (const PagePoolExhausted &) {
                    // the level-2 reserve ran out (pgR_mult has doubled): extract the range again below
                }
            }
            c->l1_live = false;      // another range, or one already built: extract again
        }
        for (int attempt = 0;; attempt++) {
            Sc1Dst d;
            if (have_pre && attempt == 0) {
                d = paged_local_dst(c);
            } else {
                d = paged_begin_local(c, n_upper, false, 1u << attempt);
                c->sc1_out_frac = c->range_all ? 1.0 : std::min(1.0, (double)n_upper / (double)n_all / 1.15);
                scatter_segments(c, P, d);
                c->sc1_out_frac = 1.0;
            }
            try {
                paged_finish(c, d, true, bin_d2, n_upper);
                break;
            } catch (const PagePoolExhausted &) {
                // a range held more instances than the hint said: take the pages it needs and go again
                if (attempt >= 3) throw;
                n_upper = std::min<uint64_t>(n_all, n_upper * 2);
            }
        }
        return;
    }
    c->blk_counts.reserve(std::max<uint64_t>(nblk, 1) * 4, c->stream);
    const uint32_t *seq = c->pool_seq.as<uint32_t>(), *bad = c->pool_bad.as<uint32_t>();
    const int range_all = c->range_all ? 1 : 0;
    c->pre_valid = false;
    uint32_t *d_counts = c->blk_counts.as<uint32_t>();
    for (auto &sg : segs) {
        if (!sg.list)
            KLAUNCH(c, "extract_count", (double)sg.nblocks * EXT_BLOCK_POS * 3 / 8,
                    (k_extract<KeyT, false, 1><<<(unsigned)sg.nblocks, EXT_THREADS, 0, c->stream>>>(
                        seq, bad, sg.begin, c->k, c->range_lo, c->range_hi, range_all, d_blk_sample,
                        d_counts + sg.blk0, nullptr, nullptr, nullptr)));
        else
            KLAUNCH(c, "list_count", (double)sg.nblocks * EXT_BLOCK_POS * sizeof(KeyT),
                    (k_list_gather<KeyT, false, 1><<<(unsigned)sg.nblocks, EXT_THREADS, 0, c->stream>>>(
                        c->list_keys.as<KeyT>(), sg.begin, c->range_lo, c->range_hi, range_all,
                        d_list_sample + (sg.blk0 - stream_blocks), d_list_valid + (sg.blk0 - stream_blocks),
                        d_counts + sg.blk0, nullptr, nullptr, nullptr)));
    }
    const uint64_t n = nblk ? scan_counts(c, d_counts, nblk, c->blk_offs) : 0;
    c->row_words = (int)round_up<int>(ceil_div<int>(c->n_samples, 32), 4);
    c->U = 0;
    c->have_union = true;
    c->n_surv = 0;
    if (n == 0) return;
    // k <= 24: one packed 64-bit record (k-mer << 16 | sample tag) per instance — half the
    // load/store/shared-memory operations per pair of the two-array layout; the sort then runs
    // on bits [16, 16 + 2k) of the record. Longer k-mers keep u64 keys + a separate u16 tag array.
    const bool packed = c->k <= 24;
    const size_t rec_bytes = packed ? 8 : sizeof(KeyT);
    c->keys_a.reserve(n * rec_bytes, c->stream);
    c->keys_b.reserve(n * rec_bytes, c->stream);
    if (!packed) {
        c->tags_a.reserve(n * 2, c->stream);
        c->tags_b.reserve(n * 2, c->stream);
    }
    const uint64_t *d_offs = (const uint64_t *)c->blk_offs.as<unsigned long long>();
    for (auto &sg : segs) {
        const double wb = (double)sg.nblocks * EXT_BLOCK_POS;
        if (!sg.list) {
            if (packed)
                KLAUNCH(c, "extract_write", wb * 3 / 8 + (double)n * 8 * sg.nblocks / nblk,
                        (k_extract<KeyT, true, 2><<<(unsigned)sg.nblocks, EXT_THREADS, 0, c->stream>>>(
                            seq, bad, sg.begin, c->k, c->range_lo, c->range_hi, range_all, d_blk_sample, nullptr,
                            d_offs + sg.blk0, c->keys_a.as<KeyT>(), nullptr)));
            else
                KLAUNCH(c, "extract_write", wb * 3 / 8 + (double)n * 10 * sg.nblocks / nblk,
                        (k_extract<KeyT, true, 1><<<(unsigned)sg.nblocks, EXT_THREADS, 0, c->stream>>>(
                            seq, bad, sg.begin, c->k, c->range_lo, c->range_hi, range_all, d_blk_sample, nullptr,
                            d_offs + sg.blk0, c->keys_a.as<KeyT>(), c->tags_a.as<uint16_t>())));
        } else {
            if (packed)
                KLAUNCH(c, "list_write", wb * sizeof(KeyT),
                        (k_list_gather<KeyT, true, 2><<<(unsigned)sg.nblocks, EXT_THREADS, 0, c->stream>>>(
                            c->list_keys.as<KeyT>(), sg.begin, c->range_lo, c->range_hi, range_all,
                            d_list_sample + (sg.blk0 - stream_blocks), d_list_valid + (sg.blk0 - stream_blocks), nullptr,
                            d_offs + sg.blk0, c->keys_a.as<KeyT>(), nullptr)));
            else
                KLAUNCH(c, "list_write", wb * sizeof(KeyT),
                        (k_list_gather<KeyT, true, 1><<<(unsigned)sg.nblocks, EXT_THREADS, 0, c->stream>>>(
                            c->list_keys.as<KeyT>(), sg.begin, c->range_lo, c->range_hi, range_all,
                            d_list_sample + (sg.blk0 - stream_blocks), d_list_valid + (sg.blk0 - stream_blocks), nullptr,
                            d_offs + sg.blk0, c->keys_a.as<KeyT>(), c->tags_a.as<uint16_t>())));
        }
    }
    const uint64_t chunks = ceil_div<uint64_t>(n, RUN_CHUNK);
    const unsigned rb = (unsigned)ceil_div<uint64_t>(chunks, RUN_THREADS / 32);
    c->blk_counts.reserve(chunks * 4, c->stream);
    if (packed) {
        sort_and_build_packed(c, c->keys_a.as<uint64_t>(), c->keys_b.as<uint64_t>(), n);
        return;
    }
    const bool in_b = radix_sort<KeyT>(c, c->keys_a.as<KeyT>(), c->keys_b.as<KeyT>(), c->tags_a.as<uint16_t>(),
                                       c->tags_b.as<uint16_t>(), n, 2 * c->k, true, 0);
    const KeyT *sk = in_b ? c->keys_b.as<KeyT>() : c->keys_a.as<KeyT>();
    const uint16_t *st = in_b ? c->tags_b.as<uint16_t>() : c->tags_a.as<uint16_t>();
    KLAUNCH(c, "run_count", (double)n * sizeof(KeyT),
            (k_run_count<KeyT><<<rb, RUN_THREADS, 0, c->stream>>>(sk, n, 0, c->blk_counts.as<uint32_t>())));
    const uint64_t U = scan_counts(c, c->blk_counts.as<uint32_t>(), chunks, c->blk_offs);
    c->U = U;
    const size_t mbytes = (size_t)U * c->row_words * 4;
    c->uni.reserve(U * 8, c->stream);
    c->matrix.reserve(mbytes + 64, c->stream);
    CK(cudaMemsetAsync(c->matrix.p, 0, mbytes, c->stream));
    KLAUNCH(c, "row_build", (double)n * (sizeof(KeyT) + 2) + (double)U * 8 + (double)mbytes,
            (k_row_build<KeyT, false><<<rb, RUN_THREADS, 0, c->stream>>>(sk, st, n, c->blk_offs.as<unsigned long long>(),
                                                                         c->uni.as<uint64_t>(), c->matrix.as<uint32_t>(),
                                                                         c->row_words)));
}

// ---------------------------------------------------------------------------------------
static void surv_reserve(ps_ctx *c, uint64_t cap) {
    c->sv_ph.reserve(cap * 4, c->stream);
    c->sv_row.reserve(cap * 8, c->stream);
    c->sv_stat.reserve(cap * 8, c->stream);
    c->sv_p.reserve(cap * 8, c->stream);
    c->sv_mx.reserve(cap * 8, c->stream);
    c->sv_my.reserve(cap * 8, c->stream);
    c->sv_n.reserve(cap * 4, c->stream);
    c->scalars.reserve(64, c->stream);
}

static SurvOut surv_out(ps_ctx *c, uint64_t cap) {
    SurvOut o;
    o.ph = c->sv_ph.as<int32_t>();
    o.row = c->sv_row.as<unsigned long long>();
    o.stat = c->sv_stat.as<double>();
    o.p = c->sv_p.as<double>();
    o.mx = c->sv_mx.as<double>();
    o.my = c->sv_my.as<double>();
    o.n_with = c->sv_n.as<uint32_t>();
    o.counter = c->scalars.as<unsigned long long>();
    o.cap = cap;
    return o;
}

static void row_mapping(const ps_ctx *c, int &wq, int &lpr_log2, int &qpl) {
    wq = c->row_words / 4;
    lpr_log2 = 0;
    while ((1 << lpr_log2) < wq && lpr_log2 < 5) lpr_log2++;
    qpl = ceil_div(wq, 1 << lpr_log2);
}

template <bool WEIGHTED, class Out>
static void launch_chi2(ps_ctx *c, int qpl, int grid, const uint4 *m, int wq, int lpr_log2, int P,
                        const uint32_t *masks, const double *totw, const int *totn, const double *w,
                        const double *wtot, int mn, int mx, double thr, Out o) {
    const double bytes = (double)c->U * c->row_words * 4;
    const bool minp = std::is_same<Out, MinpOut>::value;
    const char *nm = WEIGHTED ? (minp ? "minp_chi2_w" : "test_chi2_w") : (minp ? "minp_chi2" : "test_chi2");
    // the column masks go to shared memory when they fit the default 48 KB
    const size_t mask_bytes = (size_t)P * 2 * c->row_words * 4;
    const int sm = mask_bytes <= 40 * 1024 ? 1 : 0;
    const size_t dyn = sm ? mask_bytes : 0;
    const int N = c->n_samples;
#define PS_CHI2(Q) KLAUNCH(c, nm, bytes, (k_test_chi2<WEIGHTED, Q, Out><<<grid, 256, dyn, c->stream>>>(m, c->U, wq, lpr_log2, P, N, masks, totw, totn, w, wtot, mn, mx, thr, sm, o)))
    if (qpl <= 1) PS_CHI2(1);
    else if (qpl <= 2) PS_CHI2(2);
    else if (qpl <= 4) PS_CHI2(4);
    else PS_CHI2(16);
#undef PS_CHI2
}

template <class Out>
static void launch_chi2_sp(ps_ctx *c, int grid, const uint4 *m, int wq, int lpr_log2, int P, bool no_na,
                           const ulonglong2 *e1, const ulonglong2 *e0, int npad, const int *tot1, const int *tot0,
                           const int2 *reach, int np_lo, int np_hi, double thr, Out o) {
    const double bytes = (double)c->U * c->row_words * 4;
    const int N = c->n_samples;
    const char *nm = std::is_same<Out, MinpOut>::value ? "minp_chi2" : "test_chi2";
    if (lpr_log2 < 5) {
#define PS_CHI2SP(NN) KLAUNCH(c, nm, bytes, (k_test_chi2_sp<NN, Out><<<grid, 256, 0, c->stream>>>(m, c->U, wq, lpr_log2, P, N, e1, e0, npad, tot1, tot0, reach, np_lo, np_hi, thr, o)))
        if (no_na) PS_CHI2SP(true); else PS_CHI2SP(false);
#undef PS_CHI2SP
        return;
    }
    // rows that fill the warp: one instance per number of 32-bit words a lane owns (3..8 for 2,048 < N <= 8,190)
    const uint32_t *mw = reinterpret_cast<const uint32_t *>(m);
    const int kw = ceil_div(ceil_div(N, 32), 32), wp = c->row_words;
#define PS_CHI2SPW(K, NN) KLAUNCH(c, nm, bytes, (k_test_chi2_sp_warp<K, NN, Out><<<grid, 256, 0, c->stream>>>(mw, c->U, wp, P, N, e1, e0, npad, tot1, tot0, reach, np_lo, np_hi, thr, o)))
#define PS_CHI2SPW_K(K) case K: if (no_na) PS_CHI2SPW(K, true); else PS_CHI2SPW(K, false); break
    switch (kw) {
        PS_CHI2SPW_K(3); PS_CHI2SPW_K(4); PS_CHI2SPW_K(5); PS_CHI2SPW_K(6); PS_CHI2SPW_K(7); PS_CHI2SPW_K(8);
    default: PS_THROW(PS_ERR_ARG, "no bit-walk chi2 kernel for this row width");
    }
#undef PS_CHI2SPW_K
#undef PS_CHI2SPW
}

template <class Out>
static void launch_welch(ps_ctx *c, int qpl, int grid, const uint4 *m, int wq, int lpr_log2, int P, int N,
                         const uint32_t *nonna, const double *vals, const double *w, const double *tot,
                         const int *totn, int mn, int mx, double thr, Out o) {
    // normal quantile of the threshold: erfc(t_min / sqrt 2) = thr (bisection; thr >= 1: no screen)
    double t_min = 0.0;
    if (thr < 1.0) {
        double lo = 0.0, hi = 40.0;
        if (thr <= 0.0) lo = hi;
        for (int it = 0; it < 200 && hi - lo > 1e-12; it++) {
            const double mid = 0.5 * (lo + hi);
            if (erfc(mid * 0.70710678118654752440) > thr) lo = mid; else hi = mid;
        }
        t_min = lo * (1.0 - 1e-9);          // stay on the safe side of rounding
    }
    const double bytes = (double)c->U * c->row_words * 4;
    const char *nm = std::is_same<Out, MinpOut>::value ? "minp_welch" : "test_welch";
    if (qpl <= 1)
        KLAUNCH(c, nm, bytes, (k_test_welch<1, Out><<<grid, 256, 0, c->stream>>>(m, c->U, wq, lpr_log2, P, N, nonna, vals, w, tot, totn, mn, mx, thr, t_min, o)));
    else if (qpl <= 2)
        KLAUNCH(c, nm, bytes, (k_test_welch<2, Out><<<grid, 256, 0, c->stream>>>(m, c->U, wq, lpr_log2, P, N, nonna, vals, w, tot, totn, mn, mx, thr, t_min, o)));
    else if (qpl <= 4)
        KLAUNCH(c, nm, bytes, (k_test_welch<4, Out><<<grid, 256, 0, c->stream>>>(m, c->U, wq, lpr_log2, P, N, nonna, vals, w, tot, totn, mn, mx, thr, t_min, o)));
    else
        KLAUNCH(c, nm, bytes, (k_test_welch<16, Out><<<grid, 256, 0, c->stream>>>(m, c->U, wq, lpr_log2, P, N, nonna, vals, w, tot, totn, mn, mx, thr, t_min, o)));
}

extern "C" {

int ps_version(void) { return 100; }

int ps_ctx_create(int device, ps_ctx **out) {
    if (!out) return PS_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e);
        return PS_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { g_create_err = "device index out of range"; return PS_ERR_ARG; }
    ps_ctx *c = new ps_ctx();
    c->device = device;
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        g_create_err = std::string("cannot initialise device: ") + cudaGetErrorString(e);
        delete c;
        return PS_ERR_CUDA;
    }
    for (DevBuf *b : c->all_bufs()) b->acct = &c->dev_bytes;
    // the sort pass stages a whole tile in dynamic shared memory (up to 64 KB) next to ~19 KB
    // of static counters: opt in, and ask for the large shared-memory carve-out
#define PS_RS_ATTR(K, V, B)                                                                                   \
    cudaFuncSetAttribute(k_rs_pass<K, V, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_dyn_smem<K, V>()); \
    cudaFuncSetAttribute(k_rs_pass<K, V, B>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    PS_RS_ATTR(uint32_t, true, 8) PS_RS_ATTR(uint32_t, false, 8) PS_RS_ATTR(uint64_t, true, 8) PS_RS_ATTR(uint64_t, false, 8)
    PS_RS_ATTR(uint32_t, true, 9) PS_RS_ATTR(uint32_t, false, 9) PS_RS_ATTR(uint64_t, true, 9) PS_RS_ATTR(uint64_t, false, 9)
#undef PS_RS_ATTR
    cudaFuncSetAttribute(k_scatter1<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SC_TILE * 6 + sizeof(ScShared<SC_BINS1>)));
    cudaFuncSetAttribute(k_scatter1<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SC_TILE * 6 + sizeof(ScShared<SC_BINS1>)));
    cudaFuncSetAttribute(k_scatter1<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SC_TILE * 6 + sizeof(ScShared<SC_BINS1>)));
    cudaFuncSetAttribute(k_scatter1<0, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_scatter1<0, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_scatter1<1, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_scatter2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SC2_SMEM);
    cudaFuncSetAttribute(k_scatter2, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_bucket_build_pg<BK_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, BK_MAX_DYN_SMEM);
    cudaFuncSetAttribute(k_bucket_build_pg<BK_THREADS>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_bucket_build_pg<BK_MAX_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, BK_MAX_DYN_SMEM);
    cudaFuncSetAttribute(k_bucket_build_pg<BK_MAX_THREADS>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_mash_sketch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mash_smem(PSM_S_MAX));
    cudaFuncSetAttribute(k_mash_merge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mash_smem(PSM_S_MAX));
    cudaFuncSetAttribute(k_count_matrix<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CNT_FILTER_WORDS * 4));
    cudaFuncSetAttribute(k_count_matrix<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CNT_FILTER_WORDS * 4));
    cudaFuncSetAttribute(k_bucket_count_pg, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (const char *ev = getenv("PSKMER_SC1")) c->sc1_lean = strcmp(ev, "regs") != 0;
    if (c->sc1_lean) c->sc1_grid = 3 * PS_SMS;
    if (const char *ev = getenv("PSKMER_CHI2")) c->chi2_sparse_force = strcmp(ev, "walk") == 0;
    if (const char *ev = getenv("PSKMER_ROWS")) c->bucketed = strcmp(ev, "sorted") != 0;
    if (const char *ev = getenv("PSKMER_BK_ROW_KB")) {
        const int kb = atoi(ev);
        if (kb >= 1 && kb * 1024 + 16384 <= BK_MAX_DYN_SMEM) c->bk_row_words = kb * 256;
    }
    *out = c;
    return PS_OK;
}

void ps_ctx_destroy(ps_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (DevBuf *b : c->all_bufs()) b->release();
    for (auto &e : c->prof) {
        for (auto &pr : e.pending) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
        for (auto ev : e.pool) cudaEventDestroy(ev);
    }
    if (c->pinned) cudaFreeHost(c->pinned);
    for (auto &kv : c->ipc_open) cudaIpcCloseMemHandle(kv.second);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    cudaStreamDestroy(c->stream);
    delete c;
}

const char *ps_last_error(ps_ctx *c) { return c ? c->err.c_str() : g_create_err.c_str(); }

int ps_begin(ps_ctx *c, int k, int n_samples, uint32_t cutoff) {
    API_BEGIN(c)
    if (k < 1 || k > 32) PS_THROW(PS_ERR_ARG, "k-mer length %d outside 1..32", k);
    if (n_samples < 1 || n_samples > 65535) PS_THROW(PS_ERR_ARG, "n_samples %d outside 1..65535", n_samples);
    if (cutoff < 1) PS_THROW(PS_ERR_ARG, "cutoff must be >= 1");
    c->k = k;
    c->n_samples = n_samples;
    c->cutoff = cutoff;
    c->range_all = true;
    c->range_lo = c->range_hi = 0;
    c->samples.assign(n_samples, SampleInfo());
    c->pre_valid = false;
    c->pgA_live = false;
    c->pre_ranged = false;
    c->ing_on = false;
    c->l1_live = false;
    c->cap_hint = 0;
    c->pre_n = 0;
    c->pool_pos = 0;
    c->list_used = 0;
    c->have_union = false;
    c->U = 0;
    c->n_surv = 0;
    API_END(c)
}

int ps_set_range(ps_ctx *c, uint64_t lo, uint64_t hi) {
    API_BEGIN(c)
    c->pre_valid = false;
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (hi != 0 && hi <= lo) PS_THROW(PS_ERR_ARG, "empty k-mer range");
    c->range_lo = lo;
    c->range_hi = hi ? hi : ~0ull;
    c->range_all = (lo == 0 && hi == 0);
    c->have_union = false;
    API_END(c)
}

int ps_scatter_range(ps_ctx *c, uint64_t lo, uint64_t hi, uint64_t n_instances) {
    API_BEGIN(c)
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (!paged_ok(c)) PS_THROW(PS_ERR_ARG, "ps_scatter_range needs k = 9..16 (paged partition)");
    if (c->route_n > 1) PS_THROW(PS_ERR_STATE, "routed (multi-GPU) mode: use ps_route_scatter");
    if (hi != 0 && hi <= lo) PS_THROW(PS_ERR_ARG, "empty k-mer range");
    const uint64_t space = 1ull << (2 * c->k);
    // extraction honours the context's range: set it for the scatter, restore it afterwards
    const uint64_t keep_lo = c->range_lo, keep_hi = c->range_hi;
    const bool keep_all = c->range_all;
    {
        // the range was scattered while the samples were ingested (ps_ingest_scatter): close the open pages, done
        bool lists = false;
        for (int i = 0; i < c->n_samples; i++) lists |= c->samples[i].present && c->samples[i].list_mode;
        const uint64_t hi_n = (hi == 0 || hi >= space) ? 0 : hi, pre_hi_n = (c->pre_hi == 0 || c->pre_hi >= space) ? 0 : c->pre_hi;
        if (c->pre_valid && c->pgA_live && c->pre_ranged && !lists && c->pool_pos && c->pre_n == c->pool_pos && c->pre_lo == lo && pre_hi_n == hi_n) {
            const PagedTabs t = paged_tabs(c);
            const Sc1Dst d = paged_local_dst(c);
            KLAUNCH(c, "pg_close", 0.0, (k_pg_close1<<<c->sc1_grid, 288, 0, c->stream>>>(c->pg_state.as<ScState>(), d, 2 * c->k - 16)));
            uint32_t *h32 = reinterpret_cast<uint32_t *>(ps_pinned(c, 64));
            CK(cudaMemcpyAsync(h32, t.overflow, 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaMemcpyAsync(h32 + 1, t.cursor_a, 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            c->pre_valid = false; c->pgA_live = false; c->have_union = false;
            if (!h32[0]) {
                c->l1_instances = (uint64_t)std::min<uint32_t>(h32[1], c->pgA_cap) * PG_A;
                c->l1_live = true;
                memset(c->l1_used, 0, sizeof(c->l1_used));
                c->l1_lo = lo;
                c->l1_hi = hi_n;
                return PS_OK;
            }
            // the pool was too small for what arrived: extract again below with the usual retry
        }
    }
    c->range_lo = lo; c->range_hi = hi ? hi : ~0ull; c->range_all = (lo == 0 && hi == 0);
    c->pre_valid = false; c->pgA_live = false; c->have_union = false;
    try {
        const SegPlan P = plan_segments(c, true);
        const uint64_t n_all = P.nblk * EXT_BLOCK_POS;
        uint64_t n_upper = n_instances ? std::min<uint64_t>(n_instances, n_all) : n_all;
        const PagedTabs t = paged_tabs(c);
        for (int attempt = 0; P.nblk; attempt++) {
            const Sc1Dst d = paged_begin_local(c, n_upper, false, 1u << attempt);
            c->sc1_out_frac = c->range_all ? 1.0 : std::min(1.0, (double)n_upper / (double)n_all / 1.15);
            scatter_segments(c, P, d);
            c->sc1_out_frac = 1.0;
            KLAUNCH(c, "pg_close", 0.0, (k_pg_close1<<<c->sc1_grid, 288, 0, c->stream>>>(c->pg_state.as<ScState>(), d, 2 * c->k - 16)));
            uint32_t *h32 = reinterpret_cast<uint32_t *>(ps_pinned(c, 64));
            CK(cudaMemcpyAsync(h32, t.overflow, 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaMemcpyAsync(h32 + 1, t.cursor_a, 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            if (!h32[0]) { c->l1_instances = (uint64_t)std::min<uint32_t>(h32[1], c->pgA_cap) * PG_A; break; }
            if (attempt >= 3 || n_upper >= n_all) PS_THROW(PS_ERR_NOMEM, "level-1 page pool exhausted (%u of %u pages)", h32[1], c->pgA_cap);
            n_upper = std::min<uint64_t>(n_all, n_upper * 2);          // the range held more than the hint said
        }
        if (!P.nblk) c->l1_instances = 0;
    } catch (...) {
        c->range_lo = keep_lo; c->range_hi = keep_hi; c->range_all = keep_all;
        throw;
    }
    c->range_lo = keep_lo; c->range_hi = keep_hi; c->range_all = keep_all;
    c->l1_live = true;
    memset(c->l1_used, 0, sizeof(c->l1_used));
    c->l1_lo = lo;
    c->l1_hi = (hi == 0 || hi >= space) ? 0 : hi;
    API_END(c)
}

int ps_ingest_scatter(ps_ctx *c, uint64_t lo, uint64_t hi, uint64_t n_instances, double share) {
    API_BEGIN(c)
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (c->pool_pos) PS_THROW(PS_ERR_STATE, "ps_ingest_scatter comes before the first ps_add_samples of a job");
    if (n_instances == 0) { c->ing_on = false; return PS_OK; }
    if (!paged_ok(c)) PS_THROW(PS_ERR_ARG, "ps_ingest_scatter needs k = 9..16 (paged partition)");
    if (hi != 0 && hi <= lo) PS_THROW(PS_ERR_ARG, "empty k-mer range");
    c->ing_on = true;
    c->ing_lo = lo; c->ing_hi = hi; c->ing_n = n_instances;
    c->ing_share = share > 0.0 && share <= 1.0 ? share : 1.0;
    API_END(c)
}

int ps_set_capacity_hint(ps_ctx *c, uint64_t n_instances) {
    API_BEGIN(c)
    c->cap_hint = n_instances;
    API_END(c)
}

int ps_add_samples(ps_ctx *c, int first_idx, int count, const void *const *bytes, const size_t *lens) {
    API_BEGIN(c)
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (count < 1 || first_idx < 0 || first_idx + count > c->n_samples)
        PS_THROW(PS_ERR_ARG, "sample range [%d, %d) outside 0..%d", first_idx, first_idx + count, c->n_samples);
    if (!bytes || !lens) PS_THROW(PS_ERR_ARG, "null input table");
    for (int i = 0; i < count; i++) {
        if (c->samples[first_idx + i].present) PS_THROW(PS_ERR_STATE, "sample %d added twice", first_idx + i);
        if (lens[i] && !bytes[i]) PS_THROW(PS_ERR_ARG, "sample %d: null data", first_idx + i);
    }
    c->l1_live = false;
    if (key64(c)) add_samples_impl<uint64_t>(c, first_idx, count, bytes, lens);
    else add_samples_impl<uint32_t>(c, first_idx, count, bytes, lens);
    API_END(c)
}

int ps_sample_kmers(ps_ctx *c, int idx, uint32_t cutoff, uint64_t *kmers, uint32_t *counts, size_t cap, size_t *n) {
    API_BEGIN(c)
    if (idx < 0 || idx >= c->n_samples || !c->samples[idx].present) PS_THROW(PS_ERR_ARG, "no such sample %d", idx);
    if (!n) PS_THROW(PS_ERR_ARG, "null n");
    if (cutoff < 1) cutoff = 1;
    const uint64_t kept = key64(c) ? count_sample<uint64_t>(c, idx, cutoff) : count_sample<uint32_t>(c, idx, cutoff);
    *n = kept;
    if (kmers || counts) {
        if (cap < kept) PS_THROW(PS_ERR_ARG, "output capacity %zu < %llu", cap, (unsigned long long)kept);
        if (kept) {
            if (kmers) {
                if (key64(c)) {
                    CK(cudaMemcpyAsync(kmers, c->tmp1.p, kept * 8, cudaMemcpyDeviceToHost, c->stream));
                    CK(cudaStreamSynchronize(c->stream));
                } else {
                    std::vector<uint32_t> tmp(kept);
                    CK(cudaMemcpyAsync(tmp.data(), c->tmp1.p, kept * 4, cudaMemcpyDeviceToHost, c->stream));
                    CK(cudaStreamSynchronize(c->stream));
                    for (uint64_t i = 0; i < kept; i++) kmers[i] = tmp[i];
                }
            }
            if (counts) {
                CK(cudaMemcpyAsync(counts, c->tmp3.p, kept * 4, cudaMemcpyDeviceToHost, c->stream));
                CK(cudaStreamSynchronize(c->stream));
            }
        }
    }
    API_END(c)
}

int ps_build_union(ps_ctx *c, uint64_t *n_union) {
    API_BEGIN(c)
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (key64(c)) build_union_impl<uint64_t>(c);
    else build_union_impl<uint32_t>(c);
    if (n_union) *n_union = c->U;
    API_END(c)
}

int ps_row_words(ps_ctx *c) { return c ? (int)round_up<int>(ceil_div<int>(std::max(c->n_samples, 1), 32), 4) : PS_ERR_ARG; }

int ps_get_union(ps_ctx *c, uint64_t first, uint64_t count, uint64_t *kmers) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (first + count > c->U) PS_THROW(PS_ERR_ARG, "range beyond union size %llu", (unsigned long long)c->U);
    if (count) {
        CK(cudaMemcpyAsync(kmers, c->uni.as<uint64_t>() + first, count * 8, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    API_END(c)
}

int ps_get_rows(ps_ctx *c, uint64_t first, uint64_t count, uint32_t *rows) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (first + count > c->U) PS_THROW(PS_ERR_ARG, "range beyond union size %llu", (unsigned long long)c->U);
    if (count) {
        CK(cudaMemcpyAsync(rows, c->matrix.as<uint32_t>() + first * c->row_words, count * c->row_words * 4,
                           cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    API_END(c)
}

int ps_load_matrix(ps_ctx *c, uint64_t U, const uint64_t *kmers, const uint32_t *rows) {
    API_BEGIN(c)
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    c->row_words = (int)round_up<int>(ceil_div<int>(c->n_samples, 32), 4);
    c->U = U;
    c->have_union = true;
    c->n_surv = 0;
    if (U) {
        if (!rows) PS_THROW(PS_ERR_ARG, "null rows");
        const size_t mbytes = (size_t)U * c->row_words * 4;
        c->uni.reserve(U * 8, c->stream);
        c->matrix.reserve(mbytes + 64, c->stream);
        if (kmers) CK(cudaMemcpyAsync(c->uni.p, kmers, U * 8, cudaMemcpyDefault, c->stream));
        else CK(cudaMemsetAsync(c->uni.p, 0, U * 8, c->stream));
        CK(cudaMemcpyAsync(c->matrix.p, rows, mbytes, cudaMemcpyDefault, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    API_END(c)
}

int ps_restrict_union(ps_ctx *c, const uint64_t *db_kmers, size_t n_db, uint64_t *n_union) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (n_db && !db_kmers) PS_THROW(PS_ERR_ARG, "null database list");
    const uint64_t U = c->U;
    c->n_surv = 0;
    if (U && n_db == 0) c->U = 0;
    if (U && n_db) {
        const int wp = c->row_words;
        // the database list: used in place when it already lives on the device
        const uint64_t *d_db = db_kmers;
        cudaPointerAttributes at;
        bool on_dev = false;
        if (cudaPointerGetAttributes(&at, db_kmers) == cudaSuccess) on_dev = at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
        else cudaGetLastError();
        if (!on_dev) {
            c->tmp1.reserve(n_db * 8, c->stream);
            CK(cudaMemcpyAsync(c->tmp1.p, db_kmers, n_db * 8, cudaMemcpyHostToDevice, c->stream));
            d_db = c->tmp1.as<uint64_t>();
        }
        const uint64_t warps = ceil_div<uint64_t>(U, 32);
        const unsigned grid = (unsigned)ceil_div<uint64_t>(warps, 8);
        c->blk_counts.reserve(warps * 4, c->stream);
        const double sweep = (double)U * 8 + (double)U * 8 * 4;      // union + ~log2 probes that miss L2
        KLAUNCH(c, "kmerdb_isect", sweep,
                (k_isect<false><<<grid, 256, 0, c->stream>>>(c->uni.as<uint64_t>(), U, d_db, n_db, nullptr, wp,
                                                            c->blk_counts.as<uint32_t>(), nullptr, nullptr, nullptr)));
        const uint64_t kept = scan_counts(c, c->blk_counts.as<uint32_t>(), warps, c->blk_offs);
        c->tmp2.reserve(std::max<uint64_t>(kept, 1) * 8, c->stream);
        c->tmp3.reserve(kept * (size_t)wp * 4 + 64, c->stream);
        if (kept)
            KLAUNCH(c, "kmerdb_isect", sweep + (double)kept * (8 + 8.0 * wp),
                    (k_isect<true><<<grid, 256, 0, c->stream>>>(c->uni.as<uint64_t>(), U, d_db, n_db, c->matrix.as<uint32_t>(), wp,
                                                               nullptr, c->blk_offs.as<unsigned long long>(),
                                                               c->tmp2.as<uint64_t>(), c->tmp3.as<uint32_t>())));
        CK(cudaStreamSynchronize(c->stream));
        std::swap(c->uni, c->tmp2);
        std::swap(c->matrix, c->tmp3);
        c->U = kept;
    }
    if (n_union) *n_union = c->U;
    API_END(c)
}

}  // extern "C"

// One pass of the chi2 kernels over the matrix for P columns. minp == nullptr: the survivors (p < thr) are
// compacted, they replace those of the previous test. Otherwise the min-p epilogue lowers minp[0..P) (device,
// bit patterns of p) and the survivors of the previous test stay as they are.
static void chi2_pass(ps_ctx *c, int P, const int8_t *pheno, const double *weights, int min_samples, int max_samples,
                      double thr, unsigned long long *minp, uint64_t *n_survivors) {
    const int N = c->n_samples, wp = c->row_words;
    std::vector<uint32_t> masks((size_t)P * 2 * wp, 0);
    std::vector<double> totw((size_t)P * 2, 0.0), wtot((size_t)P * 2 * wp, 0.0);
    std::vector<int> totn(P, 0);
    for (int p = 0; p < P; p++)
        for (int s = 0; s < N; s++) {
            const int v = pheno[(size_t)p * N + s];
            const double w = weights ? weights[s] : 1.0;
            if (v == 1) { masks[((size_t)p * 2) * wp + (s >> 5)] |= 1u << (s & 31); totw[p * 2] += w; totn[p]++;
                          wtot[((size_t)p * 2) * wp + (s >> 5)] += w; }
            else if (v == 0) { masks[((size_t)p * 2 + 1) * wp + (s >> 5)] |= 1u << (s & 31); totw[p * 2 + 1] += w; totn[p]++;
                               wtot[((size_t)p * 2 + 1) * wp + (s >> 5)] += w; }
        }
    const size_t mb = masks.size() * 4;
    c->ph_masks.reserve(mb, c->stream);
    c->ph_tot.reserve(totw.size() * 8 + totn.size() * 4 + 16, c->stream);
    c->ph_vals.reserve(wtot.size() * 8, c->stream);
    CK(cudaMemcpyAsync(c->ph_vals.p, wtot.data(), wtot.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ph_masks.p, masks.data(), mb, cudaMemcpyHostToDevice, c->stream));
    double *d_totw = c->ph_tot.as<double>();
    int *d_totn = reinterpret_cast<int *>(d_totw + totw.size());
    CK(cudaMemcpyAsync(d_totw, totw.data(), totw.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d_totn, totn.data(), totn.size() * 4, cudaMemcpyHostToDevice, c->stream));
    const double *d_w = nullptr;
    if (weights) {
        std::vector<double> wpad((size_t)wp * 32, 0.0);
        for (int s = 0; s < N; s++) wpad[s] = weights[s];
        c->weights.reserve(wpad.size() * 8, c->stream);
        CK(cudaMemcpyAsync(c->weights.p, wpad.data(), wpad.size() * 8, cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        d_w = c->weights.as<double>();
    }
    // Unweighted tables: per-sample packed column membership for the bit-walk kernel (k_test_chi2_sp),
    // ten columns per pair of u64 (five 12-bit fields each). It pays once a row times the column count is large:
    // below ~512 mask words per row the masked popcounts are cheaper.
    const bool sparse_walk = !weights && N <= 8190 && (c->chi2_sparse_force || (size_t)wp * P >= 512);
    bool no_na = true;
    const ulonglong2 *d_e1 = nullptr, *d_e0 = nullptr;
    const int *d_tot1 = nullptr, *d_tot0 = nullptr;
    const int2 *d_reach = nullptr;
    int np_lo = 1, np_hi = 0;     // popcounts a row needs to be tested in some column (none: every row is skipped)
    if (sparse_walk) {
        const int npad = wp * 32, chunks = ceil_div(P, CHI2_SP_COLS);
        std::vector<unsigned long long> e((size_t)2 * chunks * npad * 2, 0ull);     // [class][chunk][sample][half]
        std::vector<int> tots((size_t)2 * P, 0);
        for (int p = 0; p < P; p++) {
            const int ch = p / CHI2_SP_COLS, j = p % CHI2_SP_COLS;
            for (int s = 0; s < N; s++) {
                const int v = pheno[(size_t)p * N + s];
                if (v != 0 && v != 1) continue;
                const int cls = v == 1 ? 0 : 1;
                e[(((size_t)cls * chunks + ch) * npad + s) * 2 + j / 5] |= 1ull << (12 * (j % 5));
                tots[(size_t)cls * P + p]++;
            }
            if (totn[p] != N) no_na = false;
        }
        // Per column, the n_with that pass the sample filter and can reach the threshold at all; a row's popcount
        // is n_with plus at most the column's NA samples. Every other row fails the kernel's screen in every column.
        std::vector<int2> reach(P);
        for (int p = 0; p < P; p++) {
            ps_chi2_reach(tots[p], tots[(size_t)P + p], min_samples, max_samples, thr, &reach[p].x, &reach[p].y);
            if (reach[p].x > reach[p].y) continue;
            const int hi = reach[p].y + (N - totn[p]);
            if (np_lo > np_hi) { np_lo = reach[p].x; np_hi = hi; }
            else { np_lo = std::min(np_lo, reach[p].x); np_hi = std::max(np_hi, hi); }
        }
        c->tmp2.reserve(e.size() * 8 + tots.size() * 4 + reach.size() * 8 + 64, c->stream);
        CK(cudaMemcpyAsync(c->tmp2.p, e.data(), e.size() * 8, cudaMemcpyHostToDevice, c->stream));
        int *dt = reinterpret_cast<int *>(c->tmp2.as<unsigned long long>() + e.size());
        CK(cudaMemcpyAsync(dt, tots.data(), tots.size() * 4, cudaMemcpyHostToDevice, c->stream));
        int2 *dr = reinterpret_cast<int2 *>(dt + tots.size());
        CK(cudaMemcpyAsync(dr, reach.data(), reach.size() * 8, cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        d_e1 = c->tmp2.as<ulonglong2>();
        d_e0 = d_e1 + (size_t)chunks * npad;
        d_tot1 = dt; d_tot0 = dt + P;
        d_reach = dr;
    }
    CK(cudaStreamSynchronize(c->stream));  // host vectors above go out of scope
    int wq, lpr_log2, qpl;
    row_mapping(c, wq, lpr_log2, qpl);
    if (minp) {
        if (qpl > 16) PS_THROW(PS_ERR_ARG, "too many samples for the test kernel (max 65535)");
        if (c->U == 0) return;
        const MinpOut o{minp};
        const int grid = PS_SMS * 8;
        if (weights) launch_chi2<true>(c, qpl, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, c->ph_masks.as<uint32_t>(), d_totw, d_totn, d_w, c->ph_vals.as<double>(), min_samples, max_samples, thr, o);
        else if (sparse_walk) launch_chi2_sp(c, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, no_na, d_e1, d_e0, wp * 32, d_tot1, d_tot0, d_reach, np_lo, np_hi, thr, o);
        else launch_chi2<false>(c, qpl, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, c->ph_masks.as<uint32_t>(), d_totw, d_totn, d_w, c->ph_vals.as<double>(), min_samples, max_samples, thr, o);
        return;
    }
    c->surv_welch = false;
    c->n_surv = 0;
    if (c->U == 0) { if (n_survivors) *n_survivors = 0; return; }
    if (qpl > 16) PS_THROW(PS_ERR_ARG, "too many samples for the test kernel (max 65535)");
    uint64_t cap = std::max<uint64_t>(c->sv_ph.cap / 4, 1u << 16);
    const int grid = PS_SMS * 8;
    for (int attempt = 0; attempt < 2; attempt++) {
        surv_reserve(c, cap);
        CK(cudaMemsetAsync(c->scalars.p, 0, 8, c->stream));
        SurvOut o = surv_out(c, cap);
        if (weights) launch_chi2<true>(c, qpl, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, c->ph_masks.as<uint32_t>(), d_totw, d_totn, d_w, c->ph_vals.as<double>(), min_samples, max_samples, thr, o);
        else if (sparse_walk) launch_chi2_sp(c, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, no_na, d_e1, d_e0, wp * 32, d_tot1, d_tot0, d_reach, np_lo, np_hi, thr, o);
        else launch_chi2<false>(c, qpl, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, c->ph_masks.as<uint32_t>(), d_totw, d_totn, d_w, c->ph_vals.as<double>(), min_samples, max_samples, thr, o);
        const uint64_t ns = ps_read_scalar<unsigned long long>(c, c->scalars.as<unsigned long long>());
        c->n_surv = ns;
        if (ns <= cap) break;
        cap = ns;
    }
    if (n_survivors) *n_survivors = c->n_surv;
}

// ps_test_welch / ps_minp_welch: one pass of k_test_welch over the matrix, as chi2_pass.
static void welch_pass(ps_ctx *c, int P, const double *pheno, const double *weights, int min_samples, int max_samples,
                       double thr, unsigned long long *minp, uint64_t *n_survivors) {
    const int N = c->n_samples, wp = c->row_words;
    const int Npad = wp * 32;
    std::vector<uint32_t> nonna((size_t)P * wp, 0);
    std::vector<double> vals((size_t)P * Npad, 0.0), tot((size_t)P * 4, 0.0);
    std::vector<int> totn(P, 0);
    for (int p = 0; p < P; p++) {
        // centre on the weighted mean of the non-NA samples: totals then subtract without cancellation
        double tw = 0, twv = 0;
        for (int s = 0; s < N; s++) {
            const double v = pheno[(size_t)p * N + s];
            if (!std::isnan(v)) { const double w = weights ? weights[s] : 1.0; tw += w; twv += w * v; totn[p]++; }
        }
        const double mu = tw > 0 ? twv / tw : 0.0;
        double cwv = 0, cwvv = 0;
        for (int s = 0; s < N; s++) {
            const double v = pheno[(size_t)p * N + s];
            if (!std::isnan(v)) {
                const double w = weights ? weights[s] : 1.0, vc = v - mu;
                nonna[(size_t)p * wp + (s >> 5)] |= 1u << (s & 31);
                vals[(size_t)p * Npad + s] = vc;
                cwv += w * vc; cwvv += w * vc * vc;
            }
        }
        tot[p * 4] = tw; tot[p * 4 + 1] = cwv; tot[p * 4 + 2] = cwvv; tot[p * 4 + 3] = mu;
    }
    c->ph_masks.reserve(nonna.size() * 4, c->stream);
    c->ph_vals.reserve(vals.size() * 8, c->stream);
    c->ph_tot.reserve(tot.size() * 8 + totn.size() * 4 + 16, c->stream);
    double *d_tot = c->ph_tot.as<double>();
    int *d_totn = reinterpret_cast<int *>(d_tot + tot.size());
    CK(cudaMemcpyAsync(d_tot, tot.data(), tot.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d_totn, totn.data(), totn.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ph_masks.p, nonna.data(), nonna.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ph_vals.p, vals.data(), vals.size() * 8, cudaMemcpyHostToDevice, c->stream));
    const double *d_w = nullptr;
    std::vector<double> wpad;
    if (weights) {
        wpad.assign((size_t)Npad, 0.0);
        for (int s = 0; s < N; s++) wpad[s] = weights[s];
        c->weights.reserve(wpad.size() * 8, c->stream);
        CK(cudaMemcpyAsync(c->weights.p, wpad.data(), wpad.size() * 8, cudaMemcpyHostToDevice, c->stream));
        d_w = c->weights.as<double>();
    }
    CK(cudaStreamSynchronize(c->stream));
    int wq, lpr_log2, qpl;
    row_mapping(c, wq, lpr_log2, qpl);
    if (minp) {
        if (qpl > 16) PS_THROW(PS_ERR_ARG, "too many samples for the test kernel (max 65535)");
        if (c->U == 0) return;
        launch_welch(c, qpl, PS_SMS * 8, c->matrix.as<uint4>(), wq, lpr_log2, P, Npad, c->ph_masks.as<uint32_t>(),
                     c->ph_vals.as<double>(), d_w, d_tot, d_totn, min_samples, max_samples, thr, MinpOut{minp});
        return;
    }
    c->surv_welch = true;
    c->n_surv = 0;
    if (c->U == 0) { if (n_survivors) *n_survivors = 0; return; }
    if (qpl > 16) PS_THROW(PS_ERR_ARG, "too many samples for the test kernel (max 65535)");
    uint64_t cap = std::max<uint64_t>(c->sv_ph.cap / 4, 1u << 16);
    const int grid = PS_SMS * 8;
    for (int attempt = 0; attempt < 2; attempt++) {
        surv_reserve(c, cap);
        CK(cudaMemsetAsync(c->scalars.p, 0, 8, c->stream));
        SurvOut o = surv_out(c, cap);
        launch_welch(c, qpl, grid, c->matrix.as<uint4>(), wq, lpr_log2, P, Npad, c->ph_masks.as<uint32_t>(),
                     c->ph_vals.as<double>(), d_w, d_tot, d_totn, min_samples, max_samples, thr, o);
        const uint64_t ns = ps_read_scalar<unsigned long long>(c, c->scalars.as<unsigned long long>());
        c->n_surv = ns;
        if (ns <= cap) break;
        cap = ns;
    }
    if (n_survivors) *n_survivors = c->n_surv;
}

// ps_minp_*: the columns in batches whose masks fit the shared-memory staging of k_test_chi2 (40 KB; whole
// groups of CHI2_SP_COLS for the bit walk), one pass over the matrix per batch, thr = 1 (no screen prunes a row).
template <class T, class Pass>
static void minp_batches(ps_ctx *c, int n_cols, const T *pheno, double *minp, Pass pass) {
    const int N = c->n_samples;
    int bs = std::max(1, (int)((40 * 1024) / ((size_t)2 * c->row_words * 4)));
    if (bs >= CHI2_SP_COLS) bs -= bs % CHI2_SP_COLS;
    c->ph_minp.reserve((size_t)n_cols * 8, c->stream);
    unsigned long long *d = c->ph_minp.as<unsigned long long>();
    std::vector<unsigned long long> one((size_t)n_cols);
    const double v1 = 1.0;
    unsigned long long b1;
    memcpy(&b1, &v1, 8);
    std::fill(one.begin(), one.end(), b1);
    CK(cudaMemcpyAsync(d, one.data(), one.size() * 8, cudaMemcpyHostToDevice, c->stream));
    for (int c0 = 0; c0 < n_cols; c0 += bs)
        pass(std::min(bs, n_cols - c0), pheno + (size_t)c0 * N, d + c0);
    CK(cudaMemcpyAsync(one.data(), d, one.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    memcpy(minp, one.data(), one.size() * 8);
}

extern "C" {

int ps_test_chi2(ps_ctx *c, int P, const int8_t *pheno, const double *weights, int min_samples, int max_samples,
                 double thr, uint64_t *n_survivors) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (P < 1 || !pheno) PS_THROW(PS_ERR_ARG, "bad phenotype table");
    chi2_pass(c, P, pheno, weights, min_samples, max_samples, thr, nullptr, n_survivors);
    API_END(c)
}

int ps_test_welch(ps_ctx *c, int P, const double *pheno, const double *weights, int min_samples, int max_samples,
                  double thr, uint64_t *n_survivors) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (P < 1 || !pheno) PS_THROW(PS_ERR_ARG, "bad phenotype table");
    welch_pass(c, P, pheno, weights, min_samples, max_samples, thr, nullptr, n_survivors);
    API_END(c)
}

int ps_minp_chi2(ps_ctx *c, int n_cols, const int8_t *pheno, const double *weights, int min_samples, int max_samples,
                 double *minp) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (n_cols < 1 || !pheno || !minp) PS_THROW(PS_ERR_ARG, "bad phenotype table");
    minp_batches(c, n_cols, pheno, minp, [&](int P, const int8_t *ph, unsigned long long *d) {
        chi2_pass(c, P, ph, weights, min_samples, max_samples, 1.0, d, nullptr);
    });
    API_END(c)
}

int ps_minp_welch(ps_ctx *c, int n_cols, const double *pheno, const double *weights, int min_samples, int max_samples,
                  double *minp) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    if (n_cols < 1 || !pheno || !minp) PS_THROW(PS_ERR_ARG, "bad phenotype table");
    minp_batches(c, n_cols, pheno, minp, [&](int P, const double *ph, unsigned long long *d) {
        welch_pass(c, P, ph, weights, min_samples, max_samples, 1.0, d, nullptr);
    });
    API_END(c)
}

int ps_select_top(ps_ctx *c, int n_pheno, uint64_t n_top, uint64_t *n_selected) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_test_* first");
    if (n_pheno < 1 || n_top < 1) PS_THROW(PS_ERR_ARG, "bad top-k request");
    const uint64_t ns = c->n_surv;
    if (ns > n_top) {        // fewer survivors than n_top overall: nothing to cut
        const int P = n_pheno;
        c->tmp2.reserve((size_t)P * 256 * 4 + (size_t)P * 8 + 64, c->stream);
        uint32_t *d_hist = c->tmp2.as<uint32_t>();
        unsigned long long *d_prefix = reinterpret_cast<unsigned long long *>(d_hist + (size_t)P * 256);
        uint8_t *hp = (uint8_t *)ps_pinned(c, (size_t)P * 256 * 4 + (size_t)P * 8 + 64);
        uint32_t *h_hist = reinterpret_cast<uint32_t *>(hp);
        unsigned long long *h_prefix = reinterpret_cast<unsigned long long *>(hp + (size_t)P * 256 * 4);
        std::vector<uint64_t> remaining(P, n_top);
        std::vector<bool> all(P, false);                   // the column has <= n_top survivors: keep everything
        for (int j = 0; j < P; j++) h_prefix[j] = 0;
        const int grid = (int)std::min<uint64_t>(PS_SMS * 8, ceil_div<uint64_t>(ns, 256));
        for (int shift = 56; shift >= 0; shift -= 8) {
            CK(cudaMemsetAsync(d_hist, 0, (size_t)P * 256 * 4, c->stream));
            CK(cudaMemcpyAsync(d_prefix, h_prefix, (size_t)P * 8, cudaMemcpyHostToDevice, c->stream));
            KLAUNCH(c, "select_top", (double)ns * 12,
                    (k_sel_hist<<<grid, 256, 0, c->stream>>>(c->sv_ph.as<int32_t>(), c->sv_p.as<double>(), ns, d_prefix, shift, d_hist)));
            CK(cudaMemcpyAsync(h_hist, d_hist, (size_t)P * 256 * 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            for (int j = 0; j < P; j++) {
                if (all[j]) continue;
                uint64_t tot = 0;
                for (int b = 0; b < 256; b++) tot += h_hist[j * 256 + b];
                if (shift == 56 && tot <= n_top) { all[j] = true; continue; }
                uint64_t cum = 0;
                int b = 0;
                for (; b < 255; b++) {
                    if (cum + h_hist[j * 256 + b] >= remaining[j]) break;
                    cum += h_hist[j * 256 + b];
                }
                remaining[j] -= cum;
                h_prefix[j] = (h_prefix[j] << 8) | (unsigned long long)b;
            }
        }
        for (int j = 0; j < P; j++) if (all[j]) h_prefix[j] = ~0ull;      // threshold: bits(p) <= prefix
        CK(cudaMemcpyAsync(d_prefix, h_prefix, (size_t)P * 8, cudaMemcpyHostToDevice, c->stream));
        // compact into a second set of arrays, then move back (ties at the threshold are all kept)
        const uint64_t cap = ns;
        c->sel_ph.reserve(cap * 4, c->stream); c->sel_row.reserve(cap * 8, c->stream); c->sel_stat.reserve(cap * 8, c->stream);
        c->sel_p.reserve(cap * 8, c->stream); c->sel_mx.reserve(cap * 8, c->stream); c->sel_my.reserve(cap * 8, c->stream);
        c->sel_n.reserve(cap * 4, c->stream);
        CK(cudaMemsetAsync(c->scalars.as<unsigned long long>() + 1, 0, 8, c->stream));
        SurvOut in = surv_out(c, ns), o;
        o.ph = c->sel_ph.as<int32_t>(); o.row = c->sel_row.as<unsigned long long>(); o.stat = c->sel_stat.as<double>();
        o.p = c->sel_p.as<double>(); o.mx = c->sel_mx.as<double>(); o.my = c->sel_my.as<double>();
        o.n_with = c->sel_n.as<uint32_t>(); o.counter = c->scalars.as<unsigned long long>() + 1; o.cap = cap;
        KLAUNCH(c, "select_top", (double)ns * 48, (k_sel_compact<<<grid, 256, 0, c->stream>>>(in, ns, d_prefix, o)));
        const uint64_t kept = ps_read_scalar<unsigned long long>(c, o.counter);
        std::swap(c->sv_ph, c->sel_ph); std::swap(c->sv_row, c->sel_row); std::swap(c->sv_stat, c->sel_stat);
        std::swap(c->sv_p, c->sel_p); std::swap(c->sv_mx, c->sel_mx); std::swap(c->sv_my, c->sel_my); std::swap(c->sv_n, c->sel_n);
        c->n_surv = kept;
    }
    if (n_selected) *n_selected = c->n_surv;
    API_END(c)
}

int ps_fetch_survivors(ps_ctx *c, size_t cap, int32_t *pheno_idx, uint64_t *row, uint64_t *kmer, double *stat,
                       double *p, double *mean_x, double *mean_y, uint32_t *n_with, uint32_t *rowbits) {
    API_BEGIN(c)
    if (!c->have_union) PS_THROW(PS_ERR_STATE, "ps_build_union first");
    const uint64_t ns = c->n_surv;
    if (cap < ns) PS_THROW(PS_ERR_ARG, "capacity %zu < %llu survivors", cap, (unsigned long long)ns);
    if (ns == 0) return PS_OK;
    const int wp = c->row_words;
    c->sv_bits.reserve(ns * wp * 4, c->stream);
    c->sv_kmer.reserve(ns * 8, c->stream);
    const int gb = (int)std::min<uint64_t>(PS_SMS * 8, ceil_div<uint64_t>(ns * wp, 256));
    KLAUNCH(c, "gather_rows", (double)ns * wp * 8,
            (k_gather_rows<<<gb, 256, 0, c->stream>>>(c->matrix.as<uint32_t>(), c->uni.as<uint64_t>(),
                                                       c->sv_row.as<unsigned long long>(), ns, wp,
                                                       c->sv_bits.as<uint32_t>(), c->sv_kmer.as<uint64_t>())));
    // one pinned landing zone, copies queued back to back, one synchronize
    const size_t a8 = round_up<size_t>(ns * 8, 64), a4 = round_up<size_t>(ns * 4, 64);
    const size_t bits_bytes = rowbits ? round_up<size_t>(ns * wp * 4, 64) : 0;
    uint8_t *hp = (uint8_t *)ps_pinned(c, 6 * a8 + 2 * a4 + bits_bytes);
    uint64_t *h_row = (uint64_t *)hp, *h_kmer = (uint64_t *)(hp + a8);
    double *h_stat = (double *)(hp + 2 * a8), *h_p = (double *)(hp + 3 * a8), *h_mx = (double *)(hp + 4 * a8),
           *h_my = (double *)(hp + 5 * a8);
    int32_t *h_ph = (int32_t *)(hp + 6 * a8);
    uint32_t *h_n = (uint32_t *)(hp + 6 * a8 + a4), *h_bits = (uint32_t *)(hp + 6 * a8 + 2 * a4);
    CK(cudaMemcpyAsync(h_ph, c->sv_ph.p, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_row, c->sv_row.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_kmer, c->sv_kmer.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_stat, c->sv_stat.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_p, c->sv_p.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_mx, c->sv_mx.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_my, c->sv_my.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_n, c->sv_n.p, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    if (rowbits) CK(cudaMemcpyAsync(h_bits, c->sv_bits.p, ns * wp * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    std::vector<uint64_t> perm(ns);
    std::iota(perm.begin(), perm.end(), 0);
    std::sort(perm.begin(), perm.end(), [&](uint64_t a, uint64_t b) {
        return h_ph[a] != h_ph[b] ? h_ph[a] < h_ph[b] : h_row[a] < h_row[b];
    });
    for (uint64_t i = 0; i < ns; i++) {
        const uint64_t j = perm[i];
        if (pheno_idx) pheno_idx[i] = h_ph[j];
        if (row) row[i] = h_row[j];
        if (kmer) kmer[i] = h_kmer[j];
        if (stat) stat[i] = h_stat[j];
        if (p) p[i] = h_p[j];
        if (mean_x) mean_x[i] = h_mx[j];
        if (mean_y) mean_y[i] = h_my[j];
        if (n_with) n_with[i] = h_n[j];
        if (rowbits) memcpy(rowbits + i * wp, h_bits + j * wp, (size_t)wp * 4);
    }
    API_END(c)
}

// Device scratch of ps_count_matrix: the counts of one chunk of samples stay under this (one row at the least)
#define CNT_CHUNK_BYTES (256ull << 20)

int ps_count_matrix(ps_ctx *c, int first_idx, int count, const uint64_t *kmers, size_t K, uint32_t *counts) {
    API_BEGIN(c)
    if (count < 1 || first_idx < 0 || (int64_t)first_idx + count > c->n_samples)
        PS_THROW(PS_ERR_ARG, "samples %d..%lld outside the job's 0..%d", first_idx, (long long)first_idx + count - 1,
                 c->n_samples - 1);
    for (int i = first_idx; i < first_idx + count; i++)
        if (!c->samples[i].present) PS_THROW(PS_ERR_ARG, "no such sample %d", i);
    if (K == 0) return PS_OK;
    if (!kmers || !counts) PS_THROW(PS_ERR_ARG, "null argument");
    if (K > (1u << 30)) PS_THROW(PS_ERR_ARG, "too many query k-mers");
    if ((size_t)count > SIZE_MAX / sizeof(uint32_t) / K) PS_THROW(PS_ERR_ARG, "count x K overflows");
    // sorted unique queries; inv maps the caller's order onto them unless the queries already ascend strictly
    std::vector<uint64_t> q;
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, kmers) == cudaSuccess && pa.type == cudaMemoryTypeDevice) {
        q.resize(K);
        CK(cudaMemcpy(q.data(), kmers, K * 8, cudaMemcpyDeviceToHost));
    } else q.assign(kmers, kmers + K);
    cudaGetLastError();
    bool identity = true;
    for (size_t j = 1; j < K && identity; j++) identity = q[j - 1] < q[j];
    std::vector<uint32_t> inv;
    if (!identity) {
        std::vector<uint64_t> u(q);
        std::sort(u.begin(), u.end());
        u.erase(std::unique(u.begin(), u.end()), u.end());
        inv.resize(K);
        for (size_t j = 0; j < K; j++) inv[j] = (uint32_t)(std::lower_bound(u.begin(), u.end(), q[j]) - u.begin());
        q.swap(u);
    }
    const uint64_t Ku = q.size();
    // radix index: qidx[t] = first query whose top bits are >= t
    const int ibits = std::min(2 * c->k, CNT_INDEX_BITS), ishift = 2 * c->k - ibits;
    std::vector<uint32_t> qidx(((size_t)1 << ibits) + 1, 0);
    for (uint64_t j = 0; j < Ku; j++) qidx[(q[j] >> ishift) + 1]++;
    for (size_t t = 1; t < qidx.size(); t++) qidx[t] += qidx[t - 1];
    c->cm_q.reserve(Ku * 8, c->stream);
    c->cm_idx.reserve(qidx.size() * 4, c->stream);
    c->cm_filter.reserve(CNT_FILTER_WORDS * 4, c->stream);
    CK(cudaMemcpyAsync(c->cm_q.p, q.data(), Ku * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->cm_idx.p, qidx.data(), qidx.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->cm_filter.p, 0, CNT_FILTER_WORDS * 4, c->stream));
    KLAUNCH(c, "count_filter", (double)Ku * 8,
            (k_count_filter<<<(unsigned)std::min<uint64_t>(PS_SMS * 4, ceil_div<uint64_t>(Ku, 256)), 256, 0, c->stream>>>(
                c->cm_q.as<uint64_t>(), Ku, c->cm_filter.as<uint32_t>())));
    if (!identity) {
        c->cm_inv.reserve(K * 4, c->stream);
        CK(cudaMemcpyAsync(c->cm_inv.p, inv.data(), K * 4, cudaMemcpyHostToDevice, c->stream));
    }
    // samples in chunks whose device counts (and their expansion to the caller's order) stay under the cap
    const uint64_t row_bytes = Ku * 4 + (identity ? 0 : (uint64_t)K * 4);
    const int chunk = (int)std::min<uint64_t>(count, std::max<uint64_t>(1, CNT_CHUNK_BYTES / row_bytes));
    c->cm_cnt.reserve((size_t)chunk * Ku * 4, c->stream);
    if (!identity) c->cm_out.reserve((size_t)chunk * K * 4, c->stream);
    c->cm_tab.reserve((size_t)chunk * 12 + 16, c->stream);
    std::vector<uint64_t> tab(chunk + (chunk + 2) / 2);   // blk_first[chunk] then blk_prefix[chunk + 1] (u32)
    for (int i0 = 0; i0 < count; i0 += chunk) {
        const int n = std::min(chunk, count - i0);
        uint32_t *prefix = reinterpret_cast<uint32_t *>(tab.data() + n);
        uint64_t blocks = 0;
        for (int i = 0; i < n; i++) {
            const SampleInfo &s = c->samples[first_idx + i0 + i];
            tab[i] = s.pos_off / EXT_BLOCK_POS;
            prefix[i] = (uint32_t)blocks;
            blocks += s.n_pos / EXT_BLOCK_POS;
        }
        if (blocks >= (1ull << 32)) PS_THROW(PS_ERR_ARG, "more than 2^32 stream blocks in one chunk");
        prefix[n] = (uint32_t)blocks;
        CK(cudaMemcpyAsync(c->cm_tab.p, tab.data(), (size_t)n * 8 + (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemsetAsync(c->cm_cnt.p, 0, (size_t)n * Ku * 4, c->stream));
        if (blocks) {
            CntArgs a;
            a.seq = c->pool_seq.as<uint32_t>(); a.bad = c->pool_bad.as<uint32_t>();
            a.blk_first = c->cm_tab.as<uint64_t>();
            a.blk_prefix = reinterpret_cast<const uint32_t *>(c->cm_tab.as<uint64_t>() + n);
            a.nrows = n; a.k = c->k;
            a.filter = c->cm_filter.as<uint32_t>();
            a.queries = c->cm_q.as<uint64_t>(); a.qidx = c->cm_idx.as<uint32_t>(); a.ishift = ishift; a.Ku = Ku;
            a.counts = c->cm_cnt.as<uint32_t>();
            const unsigned grid = (unsigned)std::min<uint64_t>(PS_SMS, ceil_div<uint64_t>(blocks * (EXT_BLOCK_POS / CNT_UNIT), CNT_THREADS / 32));
            if (key64(c))
                KLAUNCH(c, "count_matrix", (double)blocks * EXT_BLOCK_POS * 3 / 8,
                        (k_count_matrix<uint64_t><<<grid, CNT_THREADS, CNT_FILTER_WORDS * 4, c->stream>>>(a)));
            else
                KLAUNCH(c, "count_matrix", (double)blocks * EXT_BLOCK_POS * 3 / 8,
                        (k_count_matrix<uint32_t><<<grid, CNT_THREADS, CNT_FILTER_WORDS * 4, c->stream>>>(a)));
        }
        const uint32_t *res = c->cm_cnt.as<uint32_t>();
        if (!identity) {
            const uint64_t m = (uint64_t)n * K;
            KLAUNCH(c, "count_expand", (double)m * 12,
                    (k_count_expand<<<(unsigned)std::min<uint64_t>(PS_SMS * 8, ceil_div<uint64_t>(m, 256)), 256, 0, c->stream>>>(
                        res, Ku, c->cm_inv.as<uint32_t>(), K, m, c->cm_out.as<uint32_t>())));
            res = c->cm_out.as<uint32_t>();
        }
        CK(cudaMemcpyAsync(counts + (size_t)i0 * K, res, (size_t)n * K * 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    API_END(c)
}

int ps_lookup(ps_ctx *c, int idx, const uint64_t *kmers, size_t K, uint32_t *counts) {
    return ps_count_matrix(c, idx, 1, kmers, K, counts);
}

int ps_export_stream(ps_ctx *c, int idx, const void **seq, const void **bad, uint64_t *n_pos) {
    API_BEGIN(c)
    if (idx < 0 || idx >= c->n_samples || !c->samples[idx].present) PS_THROW(PS_ERR_ARG, "no such sample %d", idx);
    const SampleInfo &s = c->samples[idx];
    CK(cudaStreamSynchronize(c->stream));
    if (seq) *seq = c->pool_seq.as<uint8_t>() + s.pos_off / 4;
    if (bad) *bad = c->pool_bad.as<uint8_t>() + s.pos_off / 8;
    if (n_pos) *n_pos = s.n_pos;
    API_END(c)
}

// ---- multi-GPU routing over peer page pools (SURVEY.md 8e; replaces the all-to-all) --------------------
uint64_t ps_instances_upper(ps_ctx *c) {
    if (!c) return 0;
    uint64_t n = 0;
    for (int i = 0; i < c->n_samples; i++)
        if (c->samples[i].present) n += c->samples[i].list_mode ? c->samples[i].list_n : c->samples[i].n_pos;
    return n;
}

int ps_route_pages_needed(ps_ctx *c, int nparts, int passes, uint64_t *pages) {
    API_BEGIN(c)
    if (nparts < 1 || nparts > PART_MAX || passes < 1 || !pages) PS_THROW(PS_ERR_ARG, "nparts must be 1..%d, passes >= 1", PART_MAX);
    uint64_t npos = 0;
    for (int i = 0; i < c->n_samples; i++)
        if (c->samples[i].present)
            npos += c->samples[i].list_mode ? round_up<uint64_t>(std::max<uint64_t>(c->samples[i].list_n, 1), EXT_BLOCK_POS)
                                            : c->samples[i].n_pos;
    // a sender's records for one destination: its share with 50 % head-room, plus the pages its blocks hold open
    // or in reserve for that destination's bins
    const uint64_t share = ceil_div<uint64_t>(npos + npos / 2, (uint64_t)nparts * passes * PG_A);
    const uint64_t slack = (uint64_t)c->sc1_grid * (SC_BINS1 / nparts + 16) * (paged_groups(c) + 2);
    *pages = share + slack;
    API_END(c)
}

int ps_route_setup(ps_ctx *c, int nparts, int my_rank, const uint64_t *splitters, uint64_t pages_per_sender,
                   void **pool_ptr, void **meta_ptr) {
    API_BEGIN(c)
    if (nparts == 0) { c->route_n = 0; return PS_OK; }      // back to single-GPU builds
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (!paged_ok(c)) PS_THROW(PS_ERR_ARG, "k-mer routing needs k = 9..16 (paged partition)");
    if (nparts < 1 || nparts > PART_MAX || my_rank < 0 || my_rank >= nparts) PS_THROW(PS_ERR_ARG, "bad rank %d of %d", my_rank, nparts);
    if ((nparts > 1 && !splitters) || !pool_ptr || !meta_ptr) PS_THROW(PS_ERR_ARG, "null argument");
    const uint64_t cap = (uint64_t)nparts * pages_per_sender;
    if (pages_per_sender == 0 || cap >= (1ull << 31)) PS_THROW(PS_ERR_ARG, "bad pool size");
    const uint64_t space = 1ull << (2 * c->k);
    for (int i = 0; i + 1 < nparts; i++) {
        if (i && splitters[i] < splitters[i - 1]) PS_THROW(PS_ERR_ARG, "splitters must ascend");
        c->route_spl[i] = (uint32_t)std::min<uint64_t>(splitters[i], space - 1);
    }
    const bool same_shape = c->route_n == nparts && c->route_rank == my_rank && c->route_pages == (uint32_t)pages_per_sender;
    c->route_n = nparts; c->route_rank = my_rank; c->route_pages = (uint32_t)pages_per_sender;
    c->pre_valid = false; c->pgA_live = false; c->l1_live = false;
    paged_tabs(c);
    paged_reserve_pool(c, cap, false);
    c->pg_state.reserve((size_t)(c->sc1_grid + c->sc2_grid) * sizeof(ScState), c->stream);
    // the peers' mappings stay valid as long as nothing changed shape or moved
    if (!same_shape || c->route_pool[my_rank] != c->keys_a.p || c->route_meta[my_rank] != c->pg_meta_a.p)
        for (int d = 0; d < PART_MAX; d++) { c->route_pool[d] = nullptr; c->route_meta[d] = nullptr; }
    c->route_pool[my_rank] = c->keys_a.p; c->route_meta[my_rank] = c->pg_meta_a.p;
    *pool_ptr = c->keys_a.p; *meta_ptr = c->pg_meta_a.p;
    API_END(c)
}

int ps_route_peers(ps_ctx *c, int nparts, void *const *pool_ptrs, void *const *meta_ptrs) {
    API_BEGIN(c)
    if (nparts != c->route_n || !pool_ptrs || !meta_ptrs) PS_THROW(PS_ERR_STATE, "ps_route_setup with the same nparts first");
    for (int d = 0; d < nparts; d++) {
        if (!pool_ptrs[d] || !meta_ptrs[d]) PS_THROW(PS_ERR_ARG, "null pool of rank %d", d);
        c->route_pool[d] = pool_ptrs[d]; c->route_meta[d] = meta_ptrs[d];
    }
    if (c->route_pool[c->route_rank] != c->keys_a.p || c->route_meta[c->route_rank] != c->pg_meta_a.p)
        PS_THROW(PS_ERR_STATE, "this rank's pool moved since ps_route_setup");
    API_END(c)
}

int ps_route_connect(ps_ctx *c, int nparts, ps_ctx *const *ranks) {
    API_BEGIN(c)
    if (nparts < 1 || nparts > PART_MAX) PS_THROW(PS_ERR_ARG, "nparts must be 1..%d", PART_MAX);
    if (!ranks) PS_THROW(PS_ERR_ARG, "null rank table");
    if (nparts != c->route_n) PS_THROW(PS_ERR_STATE, "ps_route_setup with the same nparts first");
    if (ranks[c->route_rank] != c) PS_THROW(PS_ERR_ARG, "ranks[%d] must be this context", c->route_rank);
    for (int d = 0; d < nparts; d++) {
        const ps_ctx *r = ranks[d];
        if (!r) PS_THROW(PS_ERR_ARG, "null context of rank %d", d);
        if (r->route_n != nparts || r->route_rank != d)
            PS_THROW(PS_ERR_STATE, "context given as rank %d is set up as rank %d of %d", d, r->route_rank, r->route_n);
        if (!r->route_pool[d] || r->route_pool[d] != r->keys_a.p || r->route_meta[d] != r->pg_meta_a.p)
            PS_THROW(PS_ERR_STATE, "rank %d has no receive pool: ps_route_setup first", d);
    }
    // k_scatter1 stores straight into the other ranks' pools: every device among them must be reachable from
    // this one before the first ps_route_scatter (plain cudaMalloc buffers: device-level peer access covers them)
    for (int d = 0; d < nparts; d++) {
        const int dev = ranks[d]->device;
        if (dev == c->device) continue;
        int ok = 0;
        CK(cudaDeviceCanAccessPeer(&ok, c->device, dev));
        if (!ok) PS_THROW(PS_ERR_ARG, "device %d cannot access device %d (no peer access between them)", c->device, dev);
        const cudaError_t e = cudaDeviceEnablePeerAccess(dev, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else CK(e);
    }
    for (int d = 0; d < nparts; d++) { c->route_pool[d] = ranks[d]->route_pool[d]; c->route_meta[d] = ranks[d]->route_meta[d]; }
    API_END(c)
}

static void route_check(ps_ctx *c) {
    if (c->route_n < 1) PS_THROW(PS_ERR_STATE, "ps_route_setup first");
    if (c->keys_a.p != c->route_pool[c->route_rank] || (uint64_t)c->route_n * c->route_pages != c->pgA_cap)
        PS_THROW(PS_ERR_STATE, "the receive pool was reallocated by another build: call ps_route_setup again");
}

int ps_route_begin(ps_ctx *c) {
    API_BEGIN(c)
    route_check(c);
    const PagedTabs t = paged_tabs(c);
    CK(cudaMemsetAsync(c->pg_meta_a.p, 0, (size_t)c->pgA_cap * 4, c->stream));
    CK(cudaMemsetAsync(c->pg_tabs.p, 0, t.zero_bytes, c->stream));
    KLAUNCH(c, "pg_close", 0.0, (k_pg_reset_state<<<c->sc1_grid + c->sc2_grid, 288, 0, c->stream>>>(c->pg_state.as<ScState>())));
    API_END(c)
}

static Sc1Dst route_dst(ps_ctx *c) {
    const PagedTabs t = paged_tabs(c);
    Sc1Dst d;
    memset(&d, 0, sizeof(d));
    d.nparts = c->route_n;
    for (int r = 0; r < c->route_n; r++) {
        if (!c->route_pool[r]) PS_THROW(PS_ERR_STATE, "pool of rank %d unknown: ps_route_peers first", r);
        d.pool[r].recs = reinterpret_cast<uint32_t *>(c->route_pool[r]);
        d.pool[r].meta = reinterpret_cast<uint32_t *>(c->route_meta[r]);
        d.pool[r].page0 = (uint32_t)c->route_rank * c->route_pages;
        d.pool[r].cap = c->route_pages;
    }
    for (int i = 0; i + 1 < c->route_n; i++) d.spl[i] = c->route_spl[i];
    d.cursor = t.cursor_a; d.overflow = t.overflow; d.trash = t.trash;
    return d;
}

int ps_route_scatter(ps_ctx *c) {
    API_BEGIN(c)
    route_check(c);
    const SegPlan P = plan_segments(c, false);     // with ps_set_range: one pass over a super-range (splitters inside it)
    const Sc1Dst d = route_dst(c);
    scatter_segments(c, P, d);
    KLAUNCH(c, "pg_close", 0.0, (k_pg_close1<<<c->sc1_grid, 288, 0, c->stream>>>(c->pg_state.as<ScState>(), d, 2 * c->k - 16)));
    API_END(c)
}

int ps_route_build(ps_ctx *c, uint64_t *n_union, int *overflow) {
    API_BEGIN(c)
    route_check(c);
    c->row_words = (int)round_up<int>(ceil_div<int>(c->n_samples, 32), 4);
    c->U = 0; c->have_union = true; c->n_surv = 0;
    uint8_t bin_d2[512];
    for (int i = 0; i < 512; i++) bin_d2[i] = (uint8_t)std::min(std::max(i - c->route_rank, 0), 255);
    int ovf = 0;
    try {
        paged_finish(c, Sc1Dst(), false, bin_d2, (uint64_t)c->pgA_cap * PG_A);
    } catch (const PagePoolExhausted &) {
        // a sender ran out of pages on some GPU: report it, every rank must learn about it together
        ovf = 1;
    }
    if (overflow) *overflow = ovf; else if (ovf) PS_THROW(PS_ERR_NOMEM, "page pool exhausted while routing");
    if (n_union) *n_union = c->U;
    API_END(c)
}

int ps_ipc_export(ps_ctx *c, const void *dev_ptr, uint8_t handle[64]) {
    API_BEGIN(c)
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, const_cast<void *>(dev_ptr)));
    memcpy(handle, &h, 64);
    API_END(c)
}

int ps_ipc_open(ps_ctx *c, const uint8_t handle[64], void **ptr) {
    API_BEGIN(c)
    const std::string key((const char *)handle, 64);
    auto it = c->ipc_open.find(key);
    if (it == c->ipc_open.end()) {
        cudaIpcMemHandle_t h;
        memcpy(&h, handle, 64);
        void *p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        it = c->ipc_open.emplace(key, p).first;
    }
    *ptr = it->second;
    API_END(c)
}

int ps_ipc_close_all(ps_ctx *c) {
    API_BEGIN(c)
    for (auto &kv : c->ipc_open) cudaIpcCloseMemHandle(kv.second);
    c->ipc_open.clear();
    API_END(c)
}

int ps_import_streams(ps_ctx *c, int first_idx, int count, const void *seq, const void *bad,
                      const uint64_t *n_pos) {
    API_BEGIN(c)
    if (c->k == 0) PS_THROW(PS_ERR_STATE, "ps_begin first");
    if (count < 1 || first_idx < 0 || first_idx + count > c->n_samples)
        PS_THROW(PS_ERR_ARG, "sample range [%d, %d) outside 0..%d", first_idx, first_idx + count, c->n_samples);
    uint64_t total = 0;
    for (int i = 0; i < count; i++) {
        if (c->samples[first_idx + i].present) PS_THROW(PS_ERR_STATE, "sample %d added twice", first_idx + i);
        if (n_pos[i] == 0 || n_pos[i] % POS_ALIGN)
            PS_THROW(PS_ERR_ARG, "n_pos must be a positive multiple of %d", POS_ALIGN);
        total += n_pos[i];
    }
    const uint64_t pool0 = c->pool_pos, pp = pool0 + total;
    c->pool_seq.reserve(pp / 4 + 64, c->stream, true, pool0 / 4);
    c->pool_bad.reserve(pp / 8 + 64, c->stream, true, pool0 / 8);
    CK(cudaMemcpyAsync(c->pool_seq.as<uint8_t>() + pool0 / 4, seq, total / 4, cudaMemcpyDefault, c->stream));
    CK(cudaMemcpyAsync(c->pool_bad.as<uint8_t>() + pool0 / 8, bad, total / 8, cudaMemcpyDefault, c->stream));
    uint64_t off = pool0;
    for (int i = 0; i < count; i++) {
        SampleInfo &s = c->samples[first_idx + i];
        s.present = true;
        s.list_mode = false;
        s.pos_off = off;
        s.n_pos = n_pos[i];
        off += n_pos[i];
    }
    c->pool_pos = pp;
    c->have_union = false;
    c->pre_valid = false;
    if (c->cutoff > 1) {
        for (int i = 0; i < count; i++) {
            if (key64(c)) list_append<uint64_t>(c, first_idx + i, count_sample<uint64_t>(c, first_idx + i, c->cutoff));
            else list_append<uint32_t>(c, first_idx + i, count_sample<uint32_t>(c, first_idx + i, c->cutoff));
        }
    }
    CK(cudaStreamSynchronize(c->stream));   // the source buffers may be released by the caller
    API_END(c)
}

int ps_import_stream(ps_ctx *c, int idx, const void *seq, const void *bad, uint64_t n_pos) {
    return ps_import_streams(c, idx, 1, seq, bad, &n_pos);
}

int ps_sample_quantiles(ps_ctx *c, int idx, int nq, uint64_t *out) {
    API_BEGIN(c)
    if (idx < 0 || idx >= c->n_samples || !c->samples[idx].present) PS_THROW(PS_ERR_ARG, "no such sample %d", idx);
    if (nq < 2 || !out) PS_THROW(PS_ERR_ARG, "need nq >= 2 and an output array");
    const uint64_t kept = key64(c) ? count_sample<uint64_t>(c, idx, 1) : count_sample<uint32_t>(c, idx, 1);
    const size_t kb = key64(c) ? 8 : 4;
    uint8_t *h = (uint8_t *)ps_pinned(c, (size_t)nq * 8);
    memset(h, 0, (size_t)nq * 8);
    if (kept >= (uint64_t)nq) {
        for (int i = 1; i < nq; i++)
            CK(cudaMemcpyAsync(h + (size_t)i * 8, c->tmp1.as<uint8_t>() + (kept * i / nq) * kb, kb,
                               cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        for (int i = 1; i < nq; i++) {
            uint64_t v = 0;
            memcpy(&v, h + (size_t)i * 8, kb);
            out[i - 1] = v;
        }
    } else {
        const uint64_t space = c->k == 32 ? ~0ull : (1ull << (2 * c->k));
        for (int i = 1; i < nq; i++) out[i - 1] = space / nq * i;
    }
    API_END(c)
}

void *ps_stream(ps_ctx *c) { return c ? (void *)c->stream : nullptr; }
uint64_t ps_launch_count(ps_ctx *c) { return c ? c->launches : 0; }
uint64_t ps_device_bytes(ps_ctx *c) { return c ? c->dev_bytes : 0; }

int ps_profile_enable(ps_ctx *c, int on) {
    if (!c) return PS_ERR_ARG;
    if (!on && c->profiling) ps_prof_collect(c);
    c->profiling = on != 0;
    if (on && getenv("PSKMER_TRACE")) {
        if (!c->trace_ref) cudaEventCreate(&c->trace_ref);
        cudaEventRecord(c->trace_ref, c->stream);
    }
    return PS_OK;
}
int ps_profile_count(ps_ctx *c) {
    if (!c) return PS_ERR_ARG;
    ps_prof_collect(c);
    return (int)c->prof.size();
}
int ps_profile_get(ps_ctx *c, int i, const char **name, uint64_t *launches, double *total_ms, double *alg_bytes) {
    if (!c || i < 0 || i >= (int)c->prof.size()) return PS_ERR_ARG;
    ps_prof_collect(c);
    const ProfEntry &e = c->prof[i];
    if (name) *name = e.name.c_str();
    if (launches) *launches = e.launches;
    if (total_ms) *total_ms = e.ms;
    if (alg_bytes) *alg_bytes = e.alg_bytes;
    return PS_OK;
}
int ps_profile_reset(ps_ctx *c) {
    if (!c) return PS_ERR_ARG;
    ps_prof_collect(c);
    for (auto &e : c->prof) { e.launches = 0; e.ms = 0; e.alg_bytes = 0; }
    return PS_OK;
}

}  // extern "C"

// ---- -w sample weights: MinHash sketches, pair counts, neighbour joining (ps_mash.cuh) ----------------------------
int ps_mash_sketch(ps_ctx *c, int first_idx, int count, int k, int s, uint32_t seed, uint64_t *hashes,
                   uint32_t *n_hashes) {
    API_BEGIN(c)
    if (k < 1 || k > 32) PS_THROW(PS_ERR_ARG, "sketch k-mer length %d outside 1..32", k);
    if (s < 1 || s > PSM_S_MAX) PS_THROW(PS_ERR_ARG, "sketch size %d outside 1..%d", s, PSM_S_MAX);
    if (count < 1 || first_idx < 0 || first_idx + count > c->n_samples)
        PS_THROW(PS_ERR_ARG, "samples %d..%d outside the job's 0..%d", first_idx, first_idx + count - 1, c->n_samples - 1);
    if (!hashes || !n_hashes) PS_THROW(PS_ERR_ARG, "null argument");
    std::vector<uint64_t> tab(2 * (size_t)count);
    uint64_t total = 0, longest = 0;
    for (int i = 0; i < count; i++) {
        const SampleInfo &si = c->samples[first_idx + i];
        if (!si.present) PS_THROW(PS_ERR_ARG, "sample %d is not present", first_idx + i);
        tab[i] = si.pos_off;
        tab[count + i] = si.n_pos;
        total += si.n_pos;
        longest = std::max(longest, si.n_pos);
    }
    // chunks of the streams: about 16 blocks per SM over all samples, at most 1 GB of chunk lists
    uint64_t chunk = round_up<uint64_t>(std::max<uint64_t>(total / (16 * PS_SMS), 1), MASH_ROUND);
    chunk = std::min<uint64_t>(std::max<uint64_t>(chunk, 16 * MASH_ROUND), 1024 * MASH_ROUND);
    while ((uint64_t)count * ceil_div<uint64_t>(longest, chunk) * s * 8 > (1ull << 30)) chunk *= 2;
    const int n_chunks = (int)ceil_div<uint64_t>(longest, chunk);
    const int cap = mash_cap(s);
    c->mash_tab.reserve(tab.size() * 8, c->stream);
    c->mash_parts.reserve((size_t)count * n_chunks * s * 8, c->stream);
    c->mash_parts_n.reserve((size_t)count * n_chunks * 4, c->stream);
    c->mash_h.reserve((size_t)count * s * 8, c->stream);
    c->mash_n.reserve((size_t)count * 4, c->stream);
    CK(cudaMemcpyAsync(c->mash_tab.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->mash_h.p, 0, (size_t)count * s * 8, c->stream));
    const uint64_t *d_off = c->mash_tab.as<uint64_t>(), *d_npos = d_off + count;
    KLAUNCH(c, "mash_sketch", (double)total * 3 / 8,
            (k_mash_sketch<<<dim3(n_chunks, count), MASH_THREADS, mash_smem(s), c->stream>>>(
                c->pool_seq.as<uint32_t>(), c->pool_bad.as<uint32_t>(), d_off, d_npos, n_chunks, chunk, k, s, cap, seed,
                c->mash_parts.as<uint64_t>(), c->mash_parts_n.as<uint32_t>())));
    KLAUNCH(c, "mash_merge", (double)count * n_chunks * s * 8,
            (k_mash_merge<<<count, MASH_THREADS, mash_smem(s), c->stream>>>(
                c->mash_parts.as<uint64_t>(), c->mash_parts_n.as<uint32_t>(), n_chunks, s, cap, c->mash_h.as<uint64_t>(),
                c->mash_n.as<uint32_t>())));
    CK(cudaMemcpyAsync(hashes, c->mash_h.p, (size_t)count * s * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(n_hashes, c->mash_n.p, (size_t)count * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    API_END(c)
}

int ps_mash_pairs(ps_ctx *c, int n, int s, const uint64_t *hashes, const uint32_t *n_hashes, uint32_t *shared_denom) {
    API_BEGIN(c)
    if (n < 1 || n > 65535) PS_THROW(PS_ERR_ARG, "number of sketches %d outside 1..65535", n);
    if (s < 1 || s > PSM_S_MAX) PS_THROW(PS_ERR_ARG, "sketch size %d outside 1..%d", s, PSM_S_MAX);
    if (!hashes || !n_hashes || !shared_denom) PS_THROW(PS_ERR_ARG, "null argument");
    c->mash_h.reserve((size_t)n * s * 8, c->stream);
    c->mash_n.reserve((size_t)n * 4, c->stream);
    c->mash_sd.reserve((size_t)n * n * 4, c->stream);
    std::vector<uint32_t> hn(n);
    CK(cudaMemcpyAsync(hn.data(), n_hashes, (size_t)n * 4, cudaMemcpyDefault, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < n; i++)
        if (hn[i] > (uint32_t)s) PS_THROW(PS_ERR_ARG, "sketch %d holds %u hashes, more than s = %d", i, hn[i], s);
    CK(cudaMemcpyAsync(c->mash_h.p, hashes, (size_t)n * s * 8, cudaMemcpyDefault, c->stream));
    CK(cudaMemcpyAsync(c->mash_n.p, hn.data(), (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
    KLAUNCH(c, "mash_pairs", (double)n * (n + 1) / 2 * s * 8,
            (k_mash_pairs<<<dim3(ceil_div(n, 256), n), 256, (size_t)s * 8, c->stream>>>(
                c->mash_h.as<uint64_t>(), c->mash_n.as<uint32_t>(), n, s, c->mash_sd.as<uint32_t>())));
    CK(cudaMemcpyAsync(shared_denom, c->mash_sd.p, (size_t)n * n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    API_END(c)
}

int ps_neighbor_joining(ps_ctx *c, int n, const double *dm, int32_t *join, double *branch) {
    API_BEGIN(c)
    if (n < 3 || n > 65535) PS_THROW(PS_ERR_ARG, "neighbour joining needs 3..65535 taxa, got %d", n);
    if (!dm || !join || !branch) PS_THROW(PS_ERR_ARG, "null argument");
    const size_t nn = (size_t)n * n;
    std::vector<double> hd;
    const double *h = dm;
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, dm) == cudaSuccess && pa.type == cudaMemoryTypeDevice) {
        hd.resize(nn);
        CK(cudaMemcpy(hd.data(), dm, nn * 8, cudaMemcpyDeviceToHost));
        h = hd.data();
    }
    cudaGetLastError();
    for (int i = 0; i < n; i++)
        for (int j = 0; j < i; j++)
            if (!(h[(size_t)i * n + j] == h[(size_t)j * n + i]))
                PS_THROW(PS_ERR_ARG, "distance matrix is not symmetric at (%d, %d)", i, j);
    c->nj_d.reserve(nn * 8, c->stream);
    c->nj_act.reserve((size_t)2 * n * 4, c->stream);
    c->nj_nd.reserve((size_t)n * 8, c->stream);
    const int part_max = 4 * PS_SMS;
    c->nj_part.reserve((size_t)part_max * sizeof(NjBest), c->stream);
    c->nj_out.reserve((size_t)2 * n * 8 + (size_t)2 * n * 4, c->stream);
    std::vector<int> iota(n);
    std::iota(iota.begin(), iota.end(), 0);
    CK(cudaMemcpyAsync(c->nj_d.p, dm, nn * 8, cudaMemcpyDefault, c->stream));
    CK(cudaMemcpyAsync(c->nj_act.p, iota.data(), (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
    int *act = c->nj_act.as<int>(), *act_next = act + n;
    double *d_branch = c->nj_out.as<double>();
    int32_t *d_join = reinterpret_cast<int32_t *>(d_branch + 2 * (size_t)n);
    size_t ld = n;
    for (int m = n, step = 0; m > 2; m--, step++) {
        if (m >= 512 && (size_t)m * 2 <= ld) {        // most slots are dead: copy the live rows and columns together
            c->nj_d2.reserve((size_t)m * m * 8, c->stream);
            KLAUNCH(c, "nj_compact", (double)m * m * 16,
                    (k_nj_compact<<<dim3(ceil_div(m, 256), m), 256, 0, c->stream>>>(c->nj_d.as<double>(), ld, act, m,
                                                                                   c->nj_d2.as<double>())));
            std::swap(c->nj_d, c->nj_d2);
            ld = m;
            CK(cudaMemcpyAsync(act, iota.data(), (size_t)m * 4, cudaMemcpyHostToDevice, c->stream));
        }
        double *D = c->nj_d.as<double>();
        KLAUNCH(c, "nj_rowsum", (double)m * m * 8,
                (k_nj_rowsum<<<ceil_div(m, 32), 32, 0, c->stream>>>(D, ld, act, m, c->nj_nd.as<double>())));
        const int n_part = std::min(ceil_div(m - 1, 8), part_max);
        KLAUNCH(c, "nj_argmin", (double)m * (m - 1) / 2 * 8,
                (k_nj_argmin<<<n_part, 256, 0, c->stream>>>(D, ld, act, m, c->nj_nd.as<double>(), c->nj_part.as<NjBest>())));
        KLAUNCH(c, "nj_update", (double)m * 32,
                (k_nj_update<<<ceil_div(m, 256), 256, 0, c->stream>>>(D, ld, act, act_next, m, c->nj_nd.as<double>(),
                                                                      c->nj_part.as<NjBest>(), n_part, step, d_join,
                                                                      d_branch)));
        std::swap(act, act_next);
    }
    int last[2];
    CK(cudaMemcpyAsync(last, act, 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpyAsync(branch + 2 * (size_t)(n - 2), c->nj_d.as<double>() + (size_t)last[1] * ld + last[0], 8,
                       cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(branch, d_branch, (size_t)2 * (n - 2) * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(join, d_join, (size_t)2 * (n - 2) * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    API_END(c)
}
