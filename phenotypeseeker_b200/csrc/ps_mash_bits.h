// ps_mash_bits.h — the per-k-mer and per-pair arithmetic of the `-w` MinHash path (ps_mash.cuh), free of CUDA-only
// constructs so that tests/native/mash_bits_check.cpp can compile it for the host and compare it with
// phenotypeseeker_b200/weights.py.
//
// Replaces: the hash of `mash sketch` (mash 2.2 Sketch.cpp getHash: MurmurHash3_x64_128 of the canonical k-mer's
// upper-case ASCII text, first 64 bits) and the (shared, denom) count of `mash dist` (CommandDistance.cpp
// compareSketches), modeling.py:386-412.
//
// Canonical k-mers: 2 bits per base, A0 C1 G2 T3, first base most significant, canonical = min(word, reverse
// complement) — the same as kmer_at. The alphabetical order of the ASCII strings equals the numeric order of the
// words (A < C < G < T both ways), so this is mash's "alphabetically smaller strand".
#pragma once
#include <math.h>
#include <stdint.h>

#include "ps_decode_bits.h"   // PS_HD

#define PSM_S_MAX 4096

// reverse the order of the 2-bit groups of x (no complement)
PS_HD uint64_t psm_rev2_64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    x = __brevll(x);
#else
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
    x = ((x >> 8) & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
    x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
    x = (x >> 32) | (x << 32);
#endif
    return ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
}

PS_HD uint64_t psm_rotl(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }

PS_HD uint64_t psm_fmix(uint64_t k) {
    k ^= k >> 33;
    k *= 0xFF51AFD7ED558CCDull;
    k ^= k >> 33;
    k *= 0xC4CEB9FE1A85EC53ull;
    k ^= k >> 33;
    return k;
}

// four 2-bit codes in the low byte of sel4 (first base lowest) -> their ASCII letters, first base in the low byte.
// On the device one PRMT: selector nibble i = code i picks byte code of 0x54474341 ("ACGT" little-endian).
PS_HD uint32_t psm_ascii4(uint32_t nib) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(0x54474341u, 0u, nib);
#else
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) r |= (uint32_t)"ACGT"[(nib >> (4 * i)) & 3u] << (8 * i);
    return r;
#endif
}

// 8 bases (16 bits, first base in the low 2 bits) -> 8 ASCII bytes, first base in the low byte
PS_HD uint64_t psm_ascii8(uint32_t b16) {
    uint32_t x = b16 & 0xFFFFu;               // 2-bit groups -> one per nibble
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    return (uint64_t)psm_ascii4(x & 0xFFFFu) | ((uint64_t)psm_ascii4(x >> 16) << 32);
}

// the little-endian u64 word w (0..3) of the zero-padded ASCII text of a k-mer whose bases sit first-base-lowest in r
PS_HD uint64_t psm_text_word(uint64_t r, int k, int w) {
    const uint64_t t = psm_ascii8((uint32_t)(r >> (16 * w)));
    const int keep = k - 8 * w;               // bytes of this word inside the k-mer
    if (keep >= 8) return t;
    if (keep <= 0) return 0;
    return t & ((1ull << (8 * keep)) - 1ull);
}

// h1 of MurmurHash3_x64_128(text of the k-mer `canon`, seed), k = 1..32
PS_HD uint64_t psm_hash_kmer(uint64_t canon, int k, uint32_t seed) {
    const uint64_t C1 = 0x87C37B91114253D5ull, C2 = 0x4CF5AD432745937Full;
    const uint64_t r = psm_rev2_64(canon << (64 - 2 * k));
    uint64_t h1 = seed, h2 = seed;
    const int nblocks = k >> 4, tail = k & 15;
    for (int b = 0; b < nblocks; b++) {
        uint64_t k1 = psm_text_word(r, k, 2 * b), k2 = psm_text_word(r, k, 2 * b + 1);
        k1 *= C1; k1 = psm_rotl(k1, 31); k1 *= C2; h1 ^= k1;
        h1 = psm_rotl(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52DCE729ull;
        k2 *= C2; k2 = psm_rotl(k2, 33); k2 *= C1; h2 ^= k2;
        h2 = psm_rotl(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495AB5ull;
    }
    if (tail > 8) {
        uint64_t k2 = psm_text_word(r, k, 2 * nblocks + 1);
        k2 *= C2; k2 = psm_rotl(k2, 33); k2 *= C1; h2 ^= k2;
    }
    if (tail > 0) {
        uint64_t k1 = psm_text_word(r, k, 2 * nblocks);
        k1 *= C1; k1 = psm_rotl(k1, 31); k1 *= C2; h1 ^= k1;
    }
    h1 ^= (uint64_t)k; h2 ^= (uint64_t)k;
    h1 += h2; h2 += h1;
    h1 = psm_fmix(h1); h2 = psm_fmix(h2);
    return h1 + h2;
}

// canonical form of the forward 2k-bit word fw
PS_HD uint64_t psm_canonical(uint64_t fw, int k) {
    const uint64_t rc = psm_rev2_64(~fw) >> (64 - 2 * k);
    return fw < rc ? fw : rc;
}

// Python's sum() of a list of floats (CPython >= 3.12, start 0), which neighbour joining's row sums go through:
// 0 + x0, then Neumaier's compensated summation, and the compensation added at the end when it is non-zero and
// finite. Not a left-to-right sum: the two differ in the last bits for about half of all random rows.
struct PsmSum {
    double f, c;
};
PS_HD void psm_sum_first(PsmSum &s, double x) { s.f = 0.0 + x; s.c = 0.0; }
PS_HD void psm_sum_add(PsmSum &s, double x) {
    const double t = s.f + x;
    if (fabs(s.f) >= fabs(x)) s.c += (s.f - t) + x;
    else s.c += (x - t) + s.f;
    s.f = t;
}
PS_HD double psm_sum_end(const PsmSum &s) {
    const bool finite = s.c - s.c == 0.0;           // false for inf and NaN
    return (s.c != 0.0 && finite) ? s.f + s.c : s.f;
}

// (shared, denom) of two ascending distinct sketches, `mash dist`'s merge walk (weights.mash_distance): denom =
// min(s, |A u B|), shared = elements of A n B among the denom smallest of A u B. Packed as shared << 16 | denom.
PS_HD uint32_t psm_pack_sd(uint32_t shared, uint32_t denom) { return shared << 16 | denom; }

PS_HD uint32_t psm_shared_denom(const uint64_t *a, uint32_t na, const uint64_t *b, uint32_t nb, uint32_t s) {
    uint32_t i = 0, j = 0, common = 0, denom = 0;
    while (denom < s && i < na && j < nb) {
        const uint64_t x = a[i], y = b[j];
        i += x <= y;
        j += y <= x;
        common += x == y;
        denom++;
    }
    if (denom < s) {
        denom += (na - i) + (nb - j);
        if (denom > s) denom = s;
    }
    return psm_pack_sd(common, denom);
}
