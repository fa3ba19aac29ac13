// ps_decode_bits.h — the per-chunk parts of the FASTA decoder (the write pass's emit and the count pass's chunk
// summary), free of CUDA-only constructs so that tests/ can compile them for the host (tests/test_decode_bits.py,
// tests/test_decode_words.py) and compare them with the byte-at-a-time transducer on the CPU.
//
// Replaces the reader half of `glistmaker` (modeling.py:303-315) together with ps_decode.cuh.
//
// A thread owns a 64-byte chunk of text (16 words) and turns it into at most 64 codes. Instead of storing
// one code byte per position and packing afterwards, the codes are kept as two bit strings in registers —
// 2 bits per base, first base most significant (the stream's own order), and 1 break bit per position,
// first position least significant — and the finished strings are OR-ed into the tile's packed output at
// the chunk's bit offset.
//
// Every word of a chunk in sequence state goes through the same instructions, whatever its bytes are: the
// bytes are classified with word-wide (SWAR) masks, the skipped ones (newlines, CR, TAB, and the bytes outside
// the chunk's [jlo, jhi)) are squeezed out with one byte permute, and the 2-bit codes and break bits of the
// kept bytes are appended with shifts. A 60-column line puts a newline at a different word of nearly every
// lane's chunk, so a per-word choice between a four-bases path and a per-byte path would run both in every
// warp. Only a chunk that enters in header state or meets an in-range '>' (about 1 in 1000 of an assembly)
// finishes in a rolled byte loop.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PS_HD __host__ __device__ __forceinline__
#define PSD_ROLLED _Pragma("unroll 1")
#define PSD_UNROLLED _Pragma("unroll")
#else
#define PS_HD inline
#define PSD_ROLLED
#define PSD_UNROLLED
#endif

#define PSD_CODE_BREAK 4u
#define PSD_CODE_SKIP 5u

// byte -> 0..3 (A C G T/U, either case), 4 = window break, 5 = skipped (1..31)
PS_HD uint32_t psd_classify(uint32_t b) {
    if (b - 1u < 31u) return PSD_CODE_SKIP;
    const uint32_t u = b & 0xDFu;
    const uint32_t idx = u - 'A';
    const bool ok = idx < 32u && ((0x00180045u >> idx) & 1u);
    uint32_t c = (u >> 1) & 3u;
    c ^= c >> 1;
    return ok ? c : PSD_CODE_BREAK;
}

struct PsdBits {
    uint64_t sq_hi, sq_lo;   // 2 bits per code, appended at the low end (first code ends up most significant)
    uint64_t bd;             // break bit of code i at bit i
    uint32_t n;              // codes so far (<= 64)
    uint32_t s;              // transducer state: 0 sequence, 1 header
};

PS_HD void psd_append1(PsdBits &o, uint32_t code) {
    o.sq_hi = (o.sq_hi << 2) | (o.sq_lo >> 62);
    o.sq_lo = (o.sq_lo << 2) | (uint64_t)(code & 3u);
    o.bd |= (uint64_t)(code >> 2) << o.n;
    o.n++;
}

// 0x80 in every byte of v that is zero (exact: no carries between bytes)
PS_HD uint32_t psd_zero_bytes(uint32_t v) { return ~(((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v | 0x7F7F7F7Fu); }

// 0x80 in every byte of x in 1..31 (skipped in sequence state): bits 7..5 clear, bits 4..0 not all clear
PS_HD uint32_t psd_skip_bytes(uint32_t x) {
    return ((x & 0x1F1F1F1Fu) + 0x7F7F7F7Fu) & ~(x | (x << 1) | (x << 2)) & 0x80808080u;
}

// 0x80 in every byte of x that is A C G T U in either case. With bit 5 (case) ignored these are 0x41 0x43 0x47
// 0x54 0x55: bit 7 clear, bit 6 set, bit 3 clear, bit 4 set exactly when bits 2..1 are 10 (T, U), and bit 0 set
// unless bits 2..1 are 10. Each condition moves one bit of a byte to that byte's bit 7, so nothing crosses bytes.
PS_HD uint32_t psd_base_bytes(uint32_t x) {
    const uint32_t tu = (x << 5) & ~(x << 6);                       // bit 2 set, bit 1 clear
    return ~x & (x << 1) & ~(x << 4) & ~((x << 3) ^ tu) & ((x << 7) | tu) & 0x80808080u;
}

// Byte-permute selector that moves the bytes flagged in k (bit i: byte i) to the front in order and takes
// byte 4 (zero, the second operand being 0) for the rest.
PS_HD uint32_t psd_sel_of(uint32_t k) {
    uint32_t sel = 0x4444u, j = 0;
    for (uint32_t i = 0; i < 4; i++)
        if ((k >> i) & 1u) { sel = (sel & ~(0xFu << (4 * j))) | (i << (4 * j)); j++; }
    return sel;
}

#if defined(__CUDACC__)
// psd_sel_of for all 16 masks. In shared memory any mix of indices in a warp is one conflict-free access; a
// constant-memory table would serialise on the distinct indices. A kernel that calls psd_fasta_chunk fills it with
// psd_sel_init() and passes a barrier first.
__shared__ uint32_t psd_sel_tab[16];
__device__ __forceinline__ void psd_sel_init() {
    if (threadIdx.x < 16) psd_sel_tab[threadIdx.x] = psd_sel_of(threadIdx.x);
}
#endif

// The bytes of v flagged in k (bit i: byte i) moved to the front in order, zero bytes after them: one PRMT with
// the second operand 0 on the device
PS_HD uint32_t psd_compact(uint32_t v, uint32_t k) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(r) : "r"(v), "r"(psd_sel_tab[k]));
    return r;
#else
    const uint32_t sel = psd_sel_of(k);
    uint32_t r = 0;
    for (int j = 0; j < 4; j++) {
        const uint32_t i = (sel >> (4 * j)) & 7u;
        if (i < 4) r |= ((v >> (8 * i)) & 0xFFu) << (8 * j);
    }
    return r;
#endif
}

PS_HD uint32_t psd_popc(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __popc(v);
#else
    return (uint32_t)__builtin_popcount(v);
#endif
}

// upper 32 bits of (hi:lo) << s, 0 <= s < 32 (SHF.L)
PS_HD uint32_t psd_funnel_l(uint32_t lo, uint32_t hi, uint32_t s) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, s);
#else
    return (uint32_t)((((uint64_t)hi << 32) | lo) << s >> 32);
#endif
}

// Bit j of the result: byte j of the chunk lies in [jlo, jhi).
PS_HD uint64_t psd_range_bits(int jlo, int jhi) {
    const uint64_t below_hi = jhi >= 64 ? ~0ull : (1ull << jhi) - 1ull;
    const uint64_t from_lo = jlo >= 64 ? 0ull : ~0ull << jlo;
    return below_hi & from_lo;
}

// 0x80 in byte i for bit i of r4
PS_HD uint32_t psd_spread4(uint32_t r4) { return (r4 * 0x10204080u) & 0x80808080u; }

// FASTA transducer over the bytes j0..63 of a chunk, one byte at a time; bytes outside [jlo, jhi) are ignored.
// Appends to o.
PS_HD void psd_fasta_bytes(const uint32_t *w, int j0, int jlo, int jhi, PsdBits &o) {
    PSD_ROLLED
    for (int j = j0 < jlo ? jlo : j0; j < jhi; j++) {
        const uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
        if (o.s == 1u) { if (b == '\n') o.s = 0u; continue; }
        if (b == '>') { psd_append1(o, PSD_CODE_BREAK); o.s = 1u; continue; }
        const uint32_t c = psd_classify(b);
        if (c != PSD_CODE_SKIP) psd_append1(o, c);
    }
}

// FASTA transducer over the bytes [jlo, jhi) of one 64-byte chunk (16 little-endian words), starting in state
// o.s; appends to o.
PS_HD void psd_fasta_chunk(const uint32_t *w, int jlo, int jhi, PsdBits &o) {
    int q = 0;
    if (o.s == 0u) {
        uint64_t rng = psd_range_bits(jlo, jhi);
        uint32_t h1 = (uint32_t)(o.sq_hi >> 32), h0 = (uint32_t)o.sq_hi, l1 = (uint32_t)(o.sq_lo >> 32), l0 = (uint32_t)o.sq_lo;
        PSD_ROLLED
        for (; q < 16; q++, rng >>= 4) {
            const uint32_t x = w[q];
            const uint32_t in = psd_spread4((uint32_t)rng & 0xFu);          // 0x80 in the bytes in [jlo, jhi)
            if (psd_zero_bytes(x ^ 0x3E3E3E3Eu) & in) break;               // '>': the rest byte by byte
            const uint32_t keep = in & ~psd_skip_bytes(x);
            const uint32_t brk = keep & ~psd_base_bytes(x);
            const uint32_t t = (x >> 1) & 0x03030303u;
            const uint32_t c = t ^ ((t >> 1) & 0x01010101u);                // A0 C1 G2 T3 per byte
            const uint32_t bf = (brk >> 7) * 0xFFu;
            const uint32_t v = psd_compact((c & ~bf) | (bf & 0x04040404u), (keep * 0x00204081u) >> 28);
            const uint32_t n2 = 2 * psd_popc(keep);
            const uint32_t p8 = ((v & 0x03030303u) * 0x40100401u) >> 24;    // first code in the top two bits
            const uint32_t f4 = ((v & 0x04040404u) * 0x01020408u) >> 26;    // first break in bit 0
            // the 128-bit code string (h1:h0:l1:l0) shifted left by n2 bits, the new codes in the freed bits
            h1 = psd_funnel_l(h0, h1, n2);
            h0 = psd_funnel_l(l1, h0, n2);
            l1 = psd_funnel_l(l0, l1, n2);
            l0 = (l0 << n2) | (p8 >> (8 - n2));
            o.bd |= (uint64_t)f4 << o.n;
            o.n += n2 >> 1;
        }
        o.sq_hi = ((uint64_t)h1 << 32) | h0;
        o.sq_lo = ((uint64_t)l1 << 32) | l0;
    }
    psd_fasta_bytes(w, 4 * q, jlo, jhi, o);
}

// Count-pass summary (k_decode_count) of a full chunk (all 64 bytes in range) from its word masks: false when the
// chunk holds a '>', and next and cnt are then not set. The loop is unrolled so that the words stay in registers.
// The chunk is walked once as if in sequence state. An incoming header state emits nothing up to the chunk's first
// '\n' and is in sequence state right after it, like the sequence-state walk, so its count is the total minus the
// count at that '\n'. next: 2 bits per incoming state (0 sequence, 1 header; 2 and 3 are unused fixed points);
// cnt: 16 bits per incoming state.
PS_HD bool psd_fasta_count_words(const uint32_t *w, uint32_t &next, uint64_t &cnt) {
    uint32_t any_gt = 0, n = 0, n_at_nl = 0;
    bool seen_nl = false;
    PSD_UNROLLED
    for (int q = 0; q < 16; q++) {
        const uint32_t x = w[q];
        any_gt |= psd_zero_bytes(x ^ 0x3E3E3E3Eu);
        const uint32_t emit = ~psd_skip_bytes(x) & 0x80808080u;
        const uint32_t nl = psd_zero_bytes(x ^ 0x0A0A0A0Au);
        if (nl && !seen_nl) {
            seen_nl = true;
            n_at_nl = n + psd_popc(emit & ((nl & (0u - nl)) - 1u));
        }
        n += psd_popc(emit);
    }
    if (any_gt) return false;
    next = ((seen_nl ? 0u : 1u) << 2) | 0xE0u;
    cnt = (uint64_t)n | ((uint64_t)(seen_nl ? n - n_at_nl : 0u) << 16);
    return true;
}

// The same summary for any chunk and any [jlo, jhi), one byte at a time.
PS_HD void psd_fasta_count_bytes(const uint32_t *w, int jlo, int jhi, uint32_t &next, uint64_t &cnt) {
    uint32_t s = 0, n = 0, n_at_nl = 0;
    bool seen_nl = false;
    PSD_ROLLED
    for (int j = jlo; j < jhi; j++) {
        const uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
        if (s == 1u) { if (b == '\n') s = 0u; }
        else if (b == '>') { s = 1u; n++; }
        else if (psd_classify(b) != PSD_CODE_SKIP) n++;
        if (b == '\n' && !seen_nl) { seen_nl = true; n_at_nl = n; }
    }
    next = s | ((seen_nl ? s : 1u) << 2) | 0xE0u;
    cnt = (uint64_t)n | ((uint64_t)(seen_nl ? n - n_at_nl : 0u) << 16);
}

// OR the chunk's strings into packed output arrays whose position 0 is `pos0` positions before this chunk's
// first code: seq words hold 16 positions each, first position in the top bits; bad words hold 32 positions
// each, first position in bit 0. or_fn(word pointer, value) performs the (atomic) OR.
template <typename OrFn>
PS_HD void psd_place(const PsdBits &o, uint32_t pos0, uint32_t *seq_words, uint32_t *bad_words, OrFn or_fn) {
    if (o.n == 0) return;
    // left-align the 2n-bit string in 128 bits
    uint64_t hi = o.sq_hi, lo = o.sq_lo;
    const uint32_t up = 128u - 2u * o.n;                               // 0 .. 126
    if (up >= 64u) { hi = lo << (up - 64u); lo = 0; }
    else if (up) { hi = (hi << up) | (lo >> (64u - up)); lo <<= up; }
    const uint32_t S[6] = {0u, (uint32_t)(hi >> 32), (uint32_t)hi, (uint32_t)(lo >> 32), (uint32_t)lo, 0u};
    const uint32_t w0 = pos0 >> 4, sh = 2u * (pos0 & 15u);
    const uint32_t nw = (sh + 2u * o.n + 31u) >> 5;                     // words touched, <= 5
    for (uint32_t j = 0; j < 5; j++) {
        if (j >= nw) break;
        const uint32_t v = sh ? ((S[j] << (32u - sh)) | (S[j + 1] >> sh)) : S[j + 1];
        if (v) or_fn(seq_words + w0 + j, v);
    }
    if (o.bd) {
        const uint32_t b0 = pos0 >> 5, bs = pos0 & 31u;
        const uint64_t l64 = o.bd << bs;
        const uint32_t v0 = (uint32_t)l64, v1 = (uint32_t)(l64 >> 32), v2 = bs ? (uint32_t)(o.bd >> (64u - bs)) : 0u;
        if (v0) or_fn(bad_words + b0, v0);
        if (v1) or_fn(bad_words + b0 + 1, v1);
        if (v2) or_fn(bad_words + b0 + 2, v2);
    }
}
