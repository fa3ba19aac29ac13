// ps_common.cuh — context, device buffers, launch/profiling plumbing for libpskmer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>
#include <algorithm>

#include "../../include/pskmer.h"

#define PS_SMS 148  // B200

struct PsError {
    int code;
    std::string msg;
};

#define PS_THROW(code_, ...)                                  \
    do {                                                      \
        char _b[512];                                         \
        snprintf(_b, sizeof(_b), __VA_ARGS__);                \
        throw PsError{code_, std::string(_b)};                \
    } while (0)

#define CK(call)                                                                       \
    do {                                                                               \
        cudaError_t _e = (call);                                                       \
        if (_e != cudaSuccess)                                                         \
            PS_THROW(PS_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), \
                     __FILE__, __LINE__);                                              \
    } while (0)

// Grow-only device buffer: capacity survives across jobs so steady-state steps never
// call cudaMalloc.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    uint64_t *acct = nullptr;  // context-wide byte counter
    // exact: no room for growth (the page pool, sized from what the job needs). Without keep the old buffer is
    // freed before the new one is taken, so that a large buffer can be replaced by a larger one.
    void reserve(size_t bytes, cudaStream_t st, bool keep = false, size_t keep_bytes = 0, bool exact = false) {
        if (bytes <= cap) return;
        size_t ncap = exact ? bytes : bytes + bytes / 8 + 256;
        ncap = (ncap + 255) & ~size_t(255);
        if (!keep) release(st);
        void *np = nullptr;
        cudaError_t e = cudaMalloc(&np, ncap);
        if (e != cudaSuccess)
            PS_THROW(PS_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", ncap, cudaGetErrorString(e));
        if (keep && p && keep_bytes) {
            CK(cudaMemcpyAsync(np, p, keep_bytes, cudaMemcpyDeviceToDevice, st));
            CK(cudaStreamSynchronize(st));
        }
        if (p) {
            CK(cudaStreamSynchronize(st));
            cudaFree(p);
        }
        if (acct) *acct += ncap - cap;
        p = np;
        cap = ncap;
    }
    void release(cudaStream_t st = nullptr) {
        if (p && st) CK(cudaStreamSynchronize(st));
        if (p) cudaFree(p);
        if (acct) *acct -= cap;
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct ProfEntry {
    std::string name;
    uint64_t launches = 0;
    double ms = 0.0;
    double alg_bytes = 0.0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    std::vector<cudaEvent_t> pool;
};

struct SampleInfo {
    bool present = false;
    bool list_mode = false;   // per-sample counted list (FASTQ or cutoff > 1)
    uint64_t pos_off = 0;     // offset (positions, multiple of 4096) in the stream pool
    uint64_t n_pos = 0;       // padded length (positions, multiple of 4096)
    uint64_t list_off = 0;    // offset (entries) in the list pool
    uint64_t list_n = 0;
};

struct Segment { uint64_t begin; uint64_t nblocks; uint64_t blk0; bool list; };

struct ps_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // uploads that overlap with decoding
    std::string err;
    uint64_t dev_bytes = 0;
    uint64_t launches = 0;

    // job
    int k = 0;
    int n_samples = 0;
    uint32_t cutoff = 1;
    uint64_t range_lo = 0, range_hi = 0;  // hi == 0 -> unbounded
    bool range_all = true;
    std::vector<SampleInfo> samples;
    uint64_t pool_pos = 0;    // positions used in the stream pool
    uint64_t list_used = 0;   // entries used in the list pool

    // multi-GPU routing (ps_route_*): this GPU's level-1 pool is cut into route_n sub-pools of route_pages
    // pages, one per sender; peers' pools are reached through CUDA IPC mappings
    int route_n = 0, route_rank = 0;
    uint32_t route_pages = 0;
    uint32_t route_spl[8] = {0};
    void *route_pool[8] = {nullptr}, *route_meta[8] = {nullptr};
    std::map<std::string, void *> ipc_open;       // peer buffers mapped through CUDA IPC

    // records extracted while the text was still uploading (ps_add_samples, host input): valid iff
    // pre_valid and pre_n == pool_pos; any other use of the sort buffers clears pre_valid
    bool pre_valid = false;
    uint64_t pre_n = 0;

    // row construction: paged partition + bucket kernels (k = 9..16) unless PSKMER_ROWS=sorted (full sort)
    bool bucketed = true;
    int bk_row_words = 10240;   // shared-memory words of k_bucket_build's row table for ordinary buckets (PSKMER_BK_ROW_KB)

    bool sc1_lean = true;       // k_scatter1 recomputes its k-mers in the grouping phase (40 registers, 3 blocks per SM); PSKMER_SC1=regs: keeps them in registers (2 blocks per SM)
    bool chi2_sparse_force = false;   // PSKMER_CHI2=walk: the bit-walk kernel for every unweighted shape it can take (tests)

    // paged partition (ps_paged.cuh): level-1 pool = keys_a: pgA_cap pages of 4 KB, then pgR_cap level-2 reserve
    // pages of 2 KB (the other level-2 pages are the halves of level-1 pages k_scatter2 has read)
    int sc1_grid = 2 * PS_SMS, sc2_grid = 3 * PS_SMS;   // sc2_grid: k_scatter2 runs three blocks per SM (SC2_BLOCKS_PER_SM)
    uint32_t pgA_cap = 0, pgR_cap = 0;   // pages
    uint32_t pgR_mult = 1;      // reserve multiple: doubles when a build overran the reserve (kept for the context's life)
    double sc1_out_frac = 1.0;  // share of the positions whose record k_scatter1 writes (range-restricted runs): profile accounting only
    uint64_t cap_hint = 0;      // ps_set_capacity_hint: expected k-mer instances of the next build (0 = from input size)
    bool pgA_live = false;      // level-1 pool holds the records of pool positions [0, pre_n) (scattered during ingest)
    // ps_scatter_range: the level-1 pool holds every instance of the k-mers in [l1_lo, l1_hi) of all samples, pages
    // closed; builds of sub-ranges that follow level-1 bin boundaries start from it instead of extracting again
    // ps_ingest_scatter: samples are scattered for [ing_lo, ing_hi) while they are ingested (overlaps the upload)
    bool ing_on = false;
    uint64_t ing_lo = 0, ing_hi = 0, ing_n = 0;
    double ing_share = 1.0;
    bool pre_ranged = false;    // the records scattered during ingest cover [pre_lo, pre_hi) only
    uint64_t pre_lo = 0, pre_hi = 0;
    bool l1_live = false;
    uint64_t l1_lo = 0, l1_hi = 0;
    uint64_t l1_used[8] = {};   // level-1 bins whose pages a build has consumed (level-2 pages were written over them)
    uint64_t l1_instances = 0;  // records in the pool (pages x 1024, upper bound)

    // stage 2 results
    bool have_union = false;
    uint64_t U = 0;
    int row_words = 0;
    // stage 3 results
    uint64_t n_surv = 0;
    bool surv_welch = false;

    // device buffers
    DevBuf staging, tile_tab, tile_sum, file_tab;          // ingest
    DevBuf pool_seq, pool_bad;                              // 2-bit streams
    DevBuf list_keys, list_counts;                          // per-sample counted lists
    DevBuf samp_tab;                                        // per-sample table on device
    DevBuf blk_counts, blk_offs, scalars, scan_sums;        // scans
    DevBuf keys_a, keys_b, tags_a, tags_b, hist, lookback;  // sort
    DevBuf uni, matrix;                                     // union + matrix
    DevBuf ph_masks, ph_vals, ph_tot, weights;              // phenotypes
    DevBuf ph_minp;                                         // ps_minp_*: per-column minima (bit patterns)
    DevBuf sv_ph, sv_row, sv_stat, sv_p, sv_mx, sv_my, sv_n, sv_perm, sv_bits, sv_kmer;
    DevBuf sel_ph, sel_row, sel_stat, sel_p, sel_mx, sel_my, sel_n;   // ps_select_top
    DevBuf tmp1, tmp2, tmp3;
    DevBuf pg_meta_a, pg_meta_b, pg_tiles, pg_tabs, pg_state, pg_blist;   // paged partition
    DevBuf mash_tab, mash_parts, mash_parts_n, mash_h, mash_n, mash_sd;              // ps_mash_sketch / ps_mash_pairs
    DevBuf nj_d, nj_d2, nj_act, nj_nd, nj_part, nj_out;                              // ps_neighbor_joining
    DevBuf cm_q, cm_idx, cm_filter, cm_tab, cm_inv, cm_cnt, cm_out;                   // ps_count_matrix

    void *pinned = nullptr;  // small pinned scratch for readbacks
    size_t pinned_cap = 0;

    bool profiling = false;
    cudaEvent_t trace_ref = nullptr;   // PSKMER_TRACE=1: per-launch timeline on stderr (gaps between kernels)
    std::vector<ProfEntry> prof;
    std::map<std::string, int> prof_idx;

    std::vector<DevBuf *> all_bufs() {
        return {&staging, &tile_tab, &tile_sum, &file_tab, &pool_seq, &pool_bad, &list_keys,
                &list_counts, &samp_tab, &blk_counts, &blk_offs, &scalars, &scan_sums, &keys_a, &keys_b,
                &tags_a, &tags_b, &hist, &lookback, &uni, &matrix, &ph_masks, &ph_vals, &ph_tot,
                &ph_minp, &weights, &sv_ph, &sv_row, &sv_stat, &sv_p, &sv_mx, &sv_my, &sv_n, &sv_perm,
                &sv_bits, &sv_kmer, &tmp1, &tmp2, &tmp3, &pg_meta_a, &pg_meta_b, &pg_tiles,
                &pg_tabs, &pg_state, &pg_blist, &sel_ph, &sel_row, &sel_stat, &sel_p, &sel_mx, &sel_my, &sel_n,
                &mash_tab, &mash_parts, &mash_parts_n, &mash_h, &mash_n, &mash_sd, &nj_d, &nj_d2, &nj_act, &nj_nd,
                &nj_part, &nj_out, &cm_q, &cm_idx, &cm_filter, &cm_tab, &cm_inv, &cm_cnt, &cm_out};
    }
};

// ---- launch wrapper: counts launches, optional CUDA-event timing per kernel name ----
struct LaunchScope {
    ps_ctx *c;
    ProfEntry *e = nullptr;
    cudaEvent_t a = nullptr, b = nullptr;
    LaunchScope(ps_ctx *ctx, const char *name, double alg_bytes = 0.0) : c(ctx) {
        c->launches++;
        if (!c->profiling) return;
        auto it = c->prof_idx.find(name);
        int idx;
        if (it == c->prof_idx.end()) {
            idx = (int)c->prof.size();
            c->prof.emplace_back();
            c->prof.back().name = name;
            c->prof_idx[name] = idx;
        } else idx = it->second;
        e = &c->prof[idx];
        e->launches++;
        e->alg_bytes += alg_bytes;
        auto get = [&]() {
            cudaEvent_t ev;
            if (!e->pool.empty()) { ev = e->pool.back(); e->pool.pop_back(); }
            else cudaEventCreate(&ev);
            return ev;
        };
        a = get(); b = get();
        cudaEventRecord(a, c->stream);
    }
    ~LaunchScope() {
        if (!e) return;
        cudaEventRecord(b, c->stream);
        e->pending.push_back({a, b});
    }
};

static inline void ps_prof_collect(ps_ctx *c) {
    std::vector<std::pair<float, std::string>> trace;
    for (auto &e : c->prof) {
        for (auto &pr : e.pending) {
            cudaEventSynchronize(pr.second);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, pr.first, pr.second);
            e.ms += ms;
            if (c->trace_ref) {
                float t0 = 0.f;
                cudaEventElapsedTime(&t0, c->trace_ref, pr.first);
                char b[160];
                snprintf(b, sizeof(b), "%10.3f %10.3f  %s", t0, t0 + ms, e.name.c_str());
                trace.push_back({t0, std::string(b)});
            }
            e.pool.push_back(pr.first);
            e.pool.push_back(pr.second);
        }
        e.pending.clear();
    }
    if (!trace.empty()) {
        std::sort(trace.begin(), trace.end());
        float prev_end = 0.f;
        for (auto &t : trace) {
            float a = 0.f, b = 0.f;
            sscanf(t.second.c_str(), "%f %f", &a, &b);
            fprintf(stderr, "[pskmer trace] %s  gap_before=%.3f\n", t.second.c_str(), a - prev_end);
            prev_end = b;
        }
    }
}

static inline void ps_check_launch(const char *name) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) PS_THROW(PS_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e));
}

// KLAUNCH(ctx, name, alg_bytes, kernel<<<...>>>(...))
#define KLAUNCH(ctx, name, alg_bytes, ...)          \
    do {                                            \
        LaunchScope _ls(ctx, name, alg_bytes);      \
        __VA_ARGS__;                                \
        ps_check_launch(name);                      \
    } while (0)

template <typename T> static inline T ceil_div(T a, T b) { return (a + b - 1) / b; }
template <typename T> static inline T round_up(T a, T b) { return ceil_div(a, b) * b; }

// small pinned readback helper
static inline void *ps_pinned(ps_ctx *c, size_t bytes) {
    if (bytes > c->pinned_cap) {
        if (c->pinned) cudaFreeHost(c->pinned);
        size_t cap = round_up<size_t>(bytes, 4096);
        CK(cudaMallocHost(&c->pinned, cap));
        c->pinned_cap = cap;
    }
    return c->pinned;
}

template <typename T> static inline T ps_read_scalar(ps_ctx *c, const T *dptr) {
    T *h = (T *)ps_pinned(c, sizeof(T));
    CK(cudaMemcpyAsync(h, dptr, sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return *h;
}

// ---- device helpers ----
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
__device__ __forceinline__ unsigned lanemask_le() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_le;" : "=r"(m));
    return m;
}
