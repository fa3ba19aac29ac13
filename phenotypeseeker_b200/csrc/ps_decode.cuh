// ps_decode.cuh — FASTA/FASTQ text -> 2-bit packed base stream + invalid-position bitmask.
//
// Replaces the reader half of `glistmaker` (modeling.py:303-315). Reader semantics are the
// ones observed from the shipped GenomeTester4 4.2.3 binary (DESIGN.md "Reader semantics"):
// bytes before the first '>'/'@' are ignored; FASTA: '>' anywhere opens a header that ends at
// '\n', bytes 1..31 are skipped, ACGTU (either case) are bases, anything else breaks the
// window; FASTQ: strict 4-line records.
//
// The reader is a finite-state transducer (2 states for FASTA, 4 line phases for FASTQ) that
// emits at most one code per input byte. Parallelisation: every 64-byte chunk is simulated
// from every possible incoming state, giving a (next_state[4], emitted[4]) summary; summaries
// compose associatively, so a warp-shuffle scan + a short walk over tile summaries gives every
// chunk its true incoming state and output offset. Pass 1 (k_decode_count) produces tile
// summaries, k_decode_walk walks them per file, pass 2 re-simulates with the known state and packs
// 16 bases / 32 mask bits per word: k_decode_write_fasta from per-thread bit strings when a launch is
// all FASTA (ps_decode_bits.h), k_decode_write from staged code bytes when it holds FASTQ.
#pragma once
#include "ps_common.cuh"
#include "ps_decode_bits.h"

#define DEC_THREADS 256
#define DEC_CHUNK 64                         // bytes per thread: amortises the block scan
#define DEC_WORDS (DEC_CHUNK / 4)
#define DEC_TILE (DEC_THREADS * DEC_CHUNK)  // 16384 input bytes per tile
#define POS_ALIGN 4096                       // sample streams are padded to this many positions

struct FileEnt {
    uint64_t off;      // byte offset of the file in the staging buffer (16 B aligned)
    uint64_t len;      // bytes
    uint32_t tile0;    // first tile of this file
    uint32_t ntiles;   // >= 1
    uint32_t start;    // first byte that matters (index of first '>' or '@'), set by k_detect
    uint32_t fmt;      // 0 none, 1 FASTA, 2 FASTQ, set by k_detect
    uint64_t m;        // emitted codes (without final break), set by k_decode_walk
    uint64_t pool_off; // position offset of the sample stream in the pool, set by host
    uint64_t n_pos;    // padded positions, set by host
};

#define CODE_BREAK 4u
#define CODE_SKIP 5u

__device__ __forceinline__ uint32_t dec_classify(uint32_t b) {
    if (b - 1u < 31u) return CODE_SKIP;  // 1..31: LF, CR, TAB ... never break a window
    uint32_t u = b & 0xDFu;              // fold case
    uint32_t idx = u - 'A';
    bool ok = idx < 32u && ((0x00180045u >> idx) & 1u);  // A C G T U
    uint32_t c = (u >> 1) & 3u;                          // A0 C1 T2 G3
    c ^= c >> 1;                                         // A0 C1 G2 T3 (U == T)
    return ok ? c : CODE_BREAK;
}

// One transducer step. fmt 1: s in {0 seq, 1 header}; fmt 2: s = line phase 0..3.
template <typename Emit>
__device__ __forceinline__ uint32_t dec_step(uint32_t fmt, uint32_t s, uint32_t b, Emit &&emit) {
    if (fmt == 1) {
        if (s == 1) return b == '\n' ? 0u : 1u;
        if (b == '>') { emit(CODE_BREAK); return 1u; }
        uint32_t c = dec_classify(b);
        if (c != CODE_SKIP) emit(c);
        return 0u;
    } else {
        if (b == '\n') { if (s == 1) emit(CODE_BREAK); return (s + 1) & 3u; }
        if (s == 1) { uint32_t c = dec_classify(b); if (c != CODE_SKIP) emit(c); }
        return s;
    }
}

// Chunk summary: next state (2 bits x 4) and emitted count (16 bits x 4) per incoming state.
struct DecSum {
    uint32_t next;
    uint64_t cnt;
};
__device__ __forceinline__ DecSum dec_identity() { return DecSum{0xE4u, 0ull}; }
// "a then b"
__device__ __forceinline__ DecSum dec_compose(const DecSum &a, const DecSum &b) {
    DecSum r{0u, 0ull};
#pragma unroll
    for (int s = 0; s < 4; s++) {
        uint32_t ns = (a.next >> (2 * s)) & 3u;
        r.next |= ((b.next >> (2 * ns)) & 3u) << (2 * s);
        uint64_t c = ((a.cnt >> (16 * s)) & 0xFFFFull) + ((b.cnt >> (16 * ns)) & 0xFFFFull);
        r.cnt |= c << (16 * s);
    }
    return r;
}

// dec_compose for FASTA summaries: every FASTA summary maps states 0 and 1 into {0, 1} and keeps states 2 and 3 as
// fixed points with no codes, so only states 0 and 1 (the low 32 bits of cnt) are composed; the result has the same
// bits as dec_compose.
__device__ __forceinline__ DecSum dec_compose_fasta(const DecSum &a, const DecSum &b) {
    const uint32_t n0 = a.next & 3u, n1 = (a.next >> 2) & 3u;
    const uint32_t ac = (uint32_t)a.cnt, bc = (uint32_t)b.cnt;
    const uint32_t c0 = (ac & 0xFFFFu) + ((bc >> (16 * n0)) & 0xFFFFu);
    const uint32_t c1 = (ac >> 16) + ((bc >> (16 * n1)) & 0xFFFFu);
    return DecSum{((b.next >> (2 * n0)) & 3u) | (((b.next >> (2 * n1)) & 3u) << 2) | 0xE0u, (uint64_t)(c0 | (c1 << 16))};
}

__device__ __forceinline__ void dec_load_chunk(const uint8_t *file, uint64_t base, uint64_t len,
                                               uint32_t w[DEC_WORDS]) {
#pragma unroll
    for (int q = 0; q < DEC_CHUNK / 16; q++) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (base + 16 * q < len) v = *reinterpret_cast<const uint4 *>(file + base + 16 * q);
        w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
}

// Summary of one chunk (its 16 words in w) for all incoming states; only bytes in [lo, hi) count.
// One walk over the bytes is enough for every incoming state:
//  FASTA  - a full chunk without '>' (all but ~1 chunk in 1000 of an assembly): psd_fasta_count_words, word masks
//           on the words in registers; any other chunk: psd_fasta_count_bytes (ps_decode_bits.h).
//  FASTQ  - the phase of a byte is (incoming phase + newlines before it) & 3; count emissions per
//           newline-segment index q, then cnt[p] = seg[(1 - p) & 3].
// The byte-wise walks read the chunk from the thread's shared-memory row `row`, so that their loops stay rolled.
__device__ __forceinline__ DecSum dec_chunk_summary(const uint32_t w[DEC_WORDS], uint32_t *row, uint64_t base,
                                                    uint64_t lo, uint64_t hi, uint32_t fmt) {
    DecSum r{0u, 0ull};
    const int jlo = lo > base ? (int)min((uint64_t)DEC_CHUNK, lo - base) : 0;
    const int jhi = hi > base ? (int)min((uint64_t)DEC_CHUNK, hi - base) : 0;
    if (fmt == 1 && jlo == 0 && jhi == DEC_CHUNK && psd_fasta_count_words(w, r.next, r.cnt)) return r;
#pragma unroll
    for (int q = 0; q < DEC_WORDS; q++) row[q] = w[q];
    if (fmt == 1) {
        psd_fasta_count_bytes(row, jlo, jhi, r.next, r.cnt);
    } else {
        uint32_t q = 0, seg0 = 0, seg1 = 0, seg2 = 0, seg3 = 0;
#pragma unroll 1
        for (int qw = 0; qw < DEC_WORDS; qw++) {
            const uint32_t x = row[qw];
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
                const int j = 4 * qw + jj;
                const uint32_t b = (x >> (8 * jj)) & 0xFFu;
                if (j >= jlo && j < jhi) {
                    const bool nl = b == '\n';
                    const uint32_t e = (nl || dec_classify(b) != CODE_SKIP) ? 1u : 0u;   // '\n' -> BREAK
                    seg0 += (q == 0) ? e : 0u; seg1 += (q == 1) ? e : 0u;
                    seg2 += (q == 2) ? e : 0u; seg3 += (q == 3) ? e : 0u;
                    if (nl) q = (q + 1) & 3u;
                }
            }
        }
        const uint32_t seg[4] = {seg0, seg1, seg2, seg3};
#pragma unroll
        for (int p = 0; p < 4; p++) {
            r.next |= ((p + q) & 3u) << (2 * p);
            r.cnt |= (uint64_t)seg[(1 - p) & 3] << (16 * p);
        }
    }
    return r;
}

// Composition of the block's summaries in thread order, valid in thread 0. dec_compose is associative but not
// commutative: the shuffle trees combine each lane with the lanes after it, first within each warp, then over
// the warp totals in warp 0.
__device__ __forceinline__ DecSum dec_block_reduce(DecSum v, DecSum *smem /*[NW]*/) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        DecSum p;
        p.next = __shfl_down_sync(0xffffffffu, v.next, d);
        p.cnt = __shfl_down_sync(0xffffffffu, v.cnt, d);
        if (lane + d < 32u) v = dec_compose(v, p);
    }
    if (lane == 0) smem[warp] = v;
    __syncthreads();
    constexpr int NW = DEC_THREADS / 32;
    if (warp == 0) {
        v = lane < (unsigned)NW ? smem[lane] : dec_identity();
#pragma unroll
        for (int d = 1; d < NW; d <<= 1) {
            DecSum p;
            p.next = __shfl_down_sync(0xffffffffu, v.next, d);
            p.cnt = __shfl_down_sync(0xffffffffu, v.cnt, d);
            if (lane + d < (unsigned)NW) v = dec_compose(v, p);
        }
    }
    return v;
}

// Block-wide exclusive scan of summaries in thread order. Returns the exclusive prefix of
// this thread; *total = composition of the whole block (valid in all threads). FASTA: every summary of the block is
// a FASTA one (dec_compose_fasta).
template <bool FASTA = false>
__device__ __forceinline__ DecSum dec_block_scan(DecSum mine, DecSum *total, DecSum *smem /*[NW + 1]*/) {
    auto compose = [](const DecSum &a, const DecSum &b) { return FASTA ? dec_compose_fasta(a, b) : dec_compose(a, b); };
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    DecSum inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        DecSum p;
        p.next = __shfl_up_sync(0xffffffffu, inc.next, d);
        p.cnt = __shfl_up_sync(0xffffffffu, inc.cnt, d);
        if (lane >= (unsigned)d) inc = compose(p, inc);
    }
    DecSum exc;
    exc.next = __shfl_up_sync(0xffffffffu, inc.next, 1);
    exc.cnt = __shfl_up_sync(0xffffffffu, inc.cnt, 1);
    if (lane == 0) exc = dec_identity();
    constexpr int NW = DEC_THREADS / 32;
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    // warp 0 turns the warp totals into exclusive warp prefixes (+ the block total) with a shuffle scan over NW lanes
    if (warp == 0) {
        DecSum v = lane < (unsigned)NW ? smem[lane] : dec_identity();
#pragma unroll
        for (int d = 1; d < NW; d <<= 1) {
            DecSum p;
            p.next = __shfl_up_sync(0xffffffffu, v.next, d);
            p.cnt = __shfl_up_sync(0xffffffffu, v.cnt, d);
            if (lane >= (unsigned)d) v = compose(p, v);
        }
        DecSum e;
        e.next = __shfl_up_sync(0xffffffffu, v.next, 1);
        e.cnt = __shfl_up_sync(0xffffffffu, v.cnt, 1);
        if (lane == 0) e = dec_identity();
        if (lane < (unsigned)NW) smem[lane] = e;
        if (lane == NW - 1) smem[NW] = v;
    }
    __syncthreads();
    const DecSum wp = smem[warp];
    *total = smem[NW];
    return compose(wp, exc);
}

// First '>' or '@' of each file: one block per file.
__global__ void k_detect(const uint8_t *__restrict__ staging, FileEnt *__restrict__ files) {
    FileEnt &f = files[blockIdx.x];
    const uint8_t *p = staging + f.off;
    const uint64_t len = f.len;
    __shared__ unsigned long long best;
    if (threadIdx.x == 0) best = ~0ull;
    __syncthreads();
    for (uint64_t base = 0; base < len; base += (uint64_t)blockDim.x * 16) {
        uint64_t i0 = base + (uint64_t)threadIdx.x * 16;
        unsigned long long found = ~0ull;
        if (i0 < len) {
            uint4 v = *reinterpret_cast<const uint4 *>(p + i0);
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 15; j >= 0; j--) {
                uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
                if ((b == '>' || b == '@') && i0 + j < len) found = i0 + j;
            }
        }
        if (found != ~0ull) atomicMin(&best, found);
        __syncthreads();
        const bool done = best != ~0ull;
        __syncthreads();
        if (done) break;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (best == ~0ull) { f.start = (uint32_t)len; f.fmt = 0; }
        else { f.start = (uint32_t)best; f.fmt = p[best] == '>' ? 1u : 2u; }
    }
}

// a thread's shared-memory row of 16 words: stride 17, conflict-free
#define DEC_IN_STRIDE 17

// Pass 1: per-tile summaries.
__global__ void __launch_bounds__(DEC_THREADS, 6)
k_decode_count(const uint8_t *__restrict__ staging, const FileEnt *__restrict__ files,
               const uint32_t *__restrict__ tile_file, uint32_t tile_base, uint32_t *__restrict__ tile_next,
               uint64_t *__restrict__ tile_cnt, uint32_t *__restrict__ chunk_next,
               uint64_t *__restrict__ chunk_cnt) {
    __shared__ DecSum sm[DEC_THREADS / 32];
    __shared__ uint32_t s_in[DEC_THREADS * DEC_IN_STRIDE];
    const uint32_t t = blockIdx.x + tile_base;
    const FileEnt f = files[tile_file[t]];
    const uint64_t base = ((uint64_t)(t - f.tile0) * DEC_THREADS + threadIdx.x) * DEC_CHUNK;
    DecSum mine = dec_identity();
    if (f.fmt != 0 && base < f.len) {
        uint32_t w[DEC_WORDS];
        dec_load_chunk(staging + f.off, base, f.len, w);
        mine = dec_chunk_summary(w, s_in + threadIdx.x * DEC_IN_STRIDE, base, f.start, f.len, f.fmt);
    }
    // pass 2 starts from this summary instead of walking the chunk a second time
    chunk_next[(size_t)t * DEC_THREADS + threadIdx.x] = mine.next;
    chunk_cnt[(size_t)t * DEC_THREADS + threadIdx.x] = mine.cnt;
    const DecSum tot = dec_block_reduce(mine, sm);
    if (threadIdx.x == 0) { tile_next[t] = tot.next; tile_cnt[t] = tot.cnt; }
}

// Walk the tile summaries of each file: incoming state and output offset per tile.
__global__ void k_decode_walk(FileEnt *__restrict__ files, int nfiles,
                              const uint32_t *__restrict__ tile_next,
                              const uint64_t *__restrict__ tile_cnt,
                              uint32_t *__restrict__ tile_state, uint32_t *__restrict__ tile_off) {
    int fi = blockIdx.x * blockDim.x + threadIdx.x;
    if (fi >= nfiles) return;
    FileEnt &f = files[fi];
    uint32_t s = 0;
    uint64_t off = 0;
    for (uint32_t t = f.tile0; t < f.tile0 + f.ntiles; t++) {
        tile_state[t] = s;
        tile_off[t] = (uint32_t)off;
        off += (tile_cnt[t] >> (16 * s)) & 0xFFFFull;
        s = (tile_next[t] >> (2 * s)) & 3u;
    }
    f.m = off;
}

// Pass 2 for launches that hold FASTQ: emit codes with the known state, pack and store. FMT = 2: every file of the
// launch is FASTQ (or empty), so only that transducer is compiled into the 64-byte emit loop — half the kernel body
// (the generic body stalled on instruction fetch half the time); FMT = 0: mixed launch, format per file. All-FASTA
// launches take k_decode_write_fasta.
template <int FMT>
__global__ void __launch_bounds__(DEC_THREADS)
k_decode_write(const uint8_t *__restrict__ staging, const FileEnt *__restrict__ files,
               const uint32_t *__restrict__ tile_file, uint32_t tile_base,
               const uint32_t *__restrict__ tile_state, const uint32_t *__restrict__ tile_off,
               const uint32_t *__restrict__ chunk_next, const uint64_t *__restrict__ chunk_cnt,
               uint32_t *__restrict__ pool_seq, uint32_t *__restrict__ pool_bad) {
    static_assert(FMT == 0 || FMT == 2, "k_decode_write: mixed (0) or FASTQ-only (2) launches");
    __shared__ DecSum sm[DEC_THREADS / 32 + 1];
    // codes are staged at (position - first 32-position group of the tile), so that every
    // group is one aligned 32-byte span of shared memory
    __shared__ __align__(16) uint8_t codes[DEC_TILE + POS_ALIGN + 64];
    const uint32_t t = blockIdx.x + tile_base;
    const FileEnt f = files[tile_file[t]];
    const uint64_t base = ((uint64_t)(t - f.tile0) * DEC_THREADS + threadIdx.x) * DEC_CHUNK;
    const bool active = f.fmt != 0 && base < f.len;
    uint32_t w[DEC_WORDS];
    DecSum mine;
    mine.next = chunk_next[(size_t)t * DEC_THREADS + threadIdx.x];
    mine.cnt = chunk_cnt[(size_t)t * DEC_THREADS + threadIdx.x];
    if (active) dec_load_chunk(staging + f.off, base, f.len, w);
    DecSum tot;
    DecSum exc = dec_block_scan(mine, &tot, sm);
    const uint32_t s0 = tile_state[t];
    uint32_t n_codes = (uint32_t)((tot.cnt >> (16 * s0)) & 0xFFFFull);
    const uint64_t gp0 = f.pool_off + tile_off[t];
    const uint32_t lead = (uint32_t)(gp0 & 31);       // slots before the tile's first position
    const bool last = (t == f.tile0 + f.ntiles - 1);
    // final break + padding up to the padded stream length ride with the last tile
    const uint32_t extra = last ? (uint32_t)(f.pool_off + f.n_pos - (gp0 + n_codes)) : 0u;
    if (threadIdx.x < lead) codes[threadIdx.x] = 0;   // lead slots: contribute zero bits
    if (active) {
        uint32_t s = (exc.next >> (2 * s0)) & 3u;
        uint32_t o = lead + (uint32_t)((exc.cnt >> (16 * s0)) & 0xFFFFull);
        const int jlo = f.start > base ? (int)min((uint64_t)DEC_CHUNK, (uint64_t)f.start - base) : 0;
        const int jhi = f.len > base ? (int)min((uint64_t)DEC_CHUNK, f.len - base) : 0;
#pragma unroll
        for (int j = 0; j < DEC_CHUNK; j++) {
            uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
            if (j >= jlo && j < jhi) s = dec_step(FMT ? (uint32_t)FMT : f.fmt, s, b, [&](uint32_t c) { codes[o++] = (uint8_t)c; });
        }
    }
    // tail: padding breaks of the last tile, then zero slots up to the group boundary
    for (uint32_t i = threadIdx.x; i < extra + 32; i += DEC_THREADS)
        codes[lead + n_codes + i] = i < extra ? (uint8_t)CODE_BREAK : (uint8_t)0;
    n_codes += extra;
    __syncthreads();
    if (n_codes == 0) return;
    const uint64_t gp1 = gp0 + n_codes;  // exclusive
    const uint64_t g_first = gp0 >> 5, g_last = (gp1 - 1) >> 5;
    const uint4 *cv = reinterpret_cast<const uint4 *>(codes);
    for (uint64_t g = g_first + threadIdx.x; g <= g_last; g += DEC_THREADS) {
        const uint32_t gi = (uint32_t)(g - g_first);
        const uint4 a = cv[2 * gi], b4 = cv[2 * gi + 1];
        const uint32_t x[8] = {a.x, a.y, a.z, a.w, b4.x, b4.y, b4.z, b4.w};
        uint32_t seq0 = 0, seq1 = 0, bad = 0;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            // 4 codes per word: 2-bit bases gathered first-base-high, break flags first-base-low
            const uint32_t p8 = ((x[q] & 0x03030303u) * 0x40100401u) >> 24;
            const uint32_t f4 = ((((x[q] >> 2) & 0x01010101u) * 0x01020408u) >> 24) & 0xFu;
            if (q < 4) seq0 |= p8 << (24 - 8 * q);
            else seq1 |= p8 << (24 - 8 * (q - 4));
            bad |= f4 << (4 * q);
        }
        const uint64_t p0 = g << 5;
        const bool full = p0 >= gp0 && p0 + 32 <= gp1;
        if (full) {
            pool_seq[2 * g] = seq0; pool_seq[2 * g + 1] = seq1; pool_bad[g] = bad;
        } else {
            if (seq0) atomicOr(&pool_seq[2 * g], seq0);
            if (seq1) atomicOr(&pool_seq[2 * g + 1], seq1);
            if (bad) atomicOr(&pool_bad[g], bad);
        }
    }
}

// Pass 2 for launches whose files are all FASTA (or empty): the same result as the byte transducer of
// k_decode_write, built from per-thread bit strings instead of one staged code byte per position
// (ps_decode_bits.h). The chunk's 16 words go through a shared-memory row so that the word loop stays rolled — the
// byte loop's fully unrolled body for FASTA (3,984 SASS instructions) stalled on instruction fetch a third of the
// time.
#define DEC_OUT_POS (DEC_TILE + POS_ALIGN + 64)
__global__ void __launch_bounds__(DEC_THREADS)
k_decode_write_fasta(const uint8_t *__restrict__ staging, const FileEnt *__restrict__ files,
                     const uint32_t *__restrict__ tile_file, uint32_t tile_base,
                     const uint32_t *__restrict__ tile_state, const uint32_t *__restrict__ tile_off,
                     const uint32_t *__restrict__ chunk_next, const uint64_t *__restrict__ chunk_cnt,
                     uint32_t *__restrict__ pool_seq, uint32_t *__restrict__ pool_bad) {
    __shared__ DecSum sm[DEC_THREADS / 32 + 1];
    __shared__ uint32_t s_in[DEC_THREADS * DEC_IN_STRIDE];
    __shared__ uint32_t s_seq[DEC_OUT_POS / 16 + 8];
    __shared__ uint32_t s_bad[DEC_OUT_POS / 32 + 8];
    const uint32_t t = blockIdx.x + tile_base;
    const FileEnt f = files[tile_file[t]];
    const uint64_t base = ((uint64_t)(t - f.tile0) * DEC_THREADS + threadIdx.x) * DEC_CHUNK;
    const bool active = f.fmt != 0 && base < f.len;
    psd_sel_init();
    for (int i = threadIdx.x; i < DEC_OUT_POS / 16 + 8; i += DEC_THREADS) s_seq[i] = 0u;
    for (int i = threadIdx.x; i < DEC_OUT_POS / 32 + 8; i += DEC_THREADS) s_bad[i] = 0u;
    uint32_t *mine_in = s_in + threadIdx.x * DEC_IN_STRIDE;
    if (active) {
        uint32_t w[DEC_WORDS];
        dec_load_chunk(staging + f.off, base, f.len, w);
#pragma unroll
        for (int q = 0; q < DEC_WORDS; q++) mine_in[q] = w[q];
    }
    DecSum mine;
    mine.next = chunk_next[(size_t)t * DEC_THREADS + threadIdx.x];
    mine.cnt = chunk_cnt[(size_t)t * DEC_THREADS + threadIdx.x];
    DecSum tot;
    DecSum exc = dec_block_scan<true>(mine, &tot, sm);    // its barriers publish the cleared and filled tables
    const uint32_t s0 = tile_state[t];
    uint32_t n_codes = (uint32_t)((tot.cnt >> (16 * s0)) & 0xFFFFull);
    const uint64_t gp0 = f.pool_off + tile_off[t];
    const uint32_t lead = (uint32_t)(gp0 & 31);
    const bool last = (t == f.tile0 + f.ntiles - 1);
    const uint32_t extra = last ? (uint32_t)(f.pool_off + f.n_pos - (gp0 + n_codes)) : 0u;
    auto or_smem = [](uint32_t *p, uint32_t v) { atomicOr(p, v); };
    if (active) {
        PsdBits o;
        o.sq_hi = 0; o.sq_lo = 0; o.bd = 0; o.n = 0;
        o.s = (exc.next >> (2 * s0)) & 3u;
        const int jlo = f.start > base ? (int)min((uint64_t)DEC_CHUNK, (uint64_t)f.start - base) : 0;
        const int jhi = f.len > base ? (int)min((uint64_t)DEC_CHUNK, f.len - base) : 0;
        psd_fasta_chunk(mine_in, jlo, jhi, o);
        psd_place(o, lead + (uint32_t)((exc.cnt >> (16 * s0)) & 0xFFFFull), s_seq, s_bad, or_smem);
    }
    // tail of the last tile: the final break and the padding up to the padded stream length are window breaks
    for (uint32_t i = threadIdx.x; i < extra; i += DEC_THREADS) {
        const uint32_t p = lead + n_codes + i;
        atomicOr(&s_bad[p >> 5], 1u << (p & 31));
    }
    n_codes += extra;
    __syncthreads();
    if (n_codes == 0) return;
    const uint64_t gp1 = gp0 + n_codes;  // exclusive
    const uint64_t g_first = gp0 >> 5, g_last = (gp1 - 1) >> 5;
    for (uint64_t g = g_first + threadIdx.x; g <= g_last; g += DEC_THREADS) {
        const uint32_t gi = (uint32_t)(g - g_first);
        const uint32_t seq0 = s_seq[2 * gi], seq1 = s_seq[2 * gi + 1], bad = s_bad[gi];
        const uint64_t p0 = g << 5;
        const bool full = p0 >= gp0 && p0 + 32 <= gp1;
        if (full) {
            pool_seq[2 * g] = seq0; pool_seq[2 * g + 1] = seq1; pool_bad[g] = bad;
        } else {
            if (seq0) atomicOr(&pool_seq[2 * g], seq0);
            if (seq1) atomicOr(&pool_seq[2 * g + 1], seq1);
            if (bad) atomicOr(&pool_bad[g], bad);
        }
    }
}
