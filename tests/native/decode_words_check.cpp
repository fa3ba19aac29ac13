// Host check of the word-wide FASTA reader in phenotypeseeker_b200/csrc/ps_decode_bits.h: the byte masks, the write
// pass's word step (psd_fasta_chunk + psd_place) and the count pass's chunk summaries (psd_fasta_count_words,
// psd_fasta_count_bytes), against a byte-at-a-time reader written here from the documented semantics (DESIGN.md
// "Reader semantics"). Built and run by tests/test_decode_words.py.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../phenotypeseeker_b200/csrc/ps_decode_bits.h"

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint32_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (uint32_t)(rng_state >> 11); }

static int failures = 0;
#define CHECK(cond, ...) do { if (!(cond)) { if (failures++ < 20) { fprintf(stderr, __VA_ARGS__); fputc('\n', stderr); } } } while (0)

// 0..3 = A C G T (U reads as T), 4 = window break, 5 = skipped
static uint32_t ref_class(uint32_t b) {
    if (b >= 1 && b <= 31) return 5;
    switch (b) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': case 'U': case 'u': return 3;
    }
    return 4;
}

// FASTA reader from state s over p[lo, hi): '>' emits a break and opens a header that ends at '\n'
static uint32_t ref_run(const uint8_t *p, int lo, int hi, uint32_t s, std::vector<uint8_t> *codes) {
    for (int i = lo; i < hi; i++) {
        const uint32_t b = p[i];
        if (s == 1) { if (b == '\n') s = 0; continue; }
        if (b == '>') { codes->push_back(4); s = 1; continue; }
        const uint32_t c = ref_class(b);
        if (c != 5) codes->push_back((uint8_t)c);
    }
    return s;
}

static void load_words(const uint8_t *p, uint32_t w[16]) { memcpy(w, p, 64); }

// psd_classify, psd_skip_bytes and psd_base_bytes for every byte value at every byte of a word
static void check_masks() {
    for (uint32_t b = 0; b < 256; b++) {
        CHECK(psd_classify(b) == ref_class(b), "psd_classify(%u) = %u", b, psd_classify(b));
        for (int pos = 0; pos < 4; pos++)
            for (int rep = 0; rep < 64; rep++) {
                uint32_t x = rnd();
                x = (x & ~(0xFFu << (8 * pos))) | (b << (8 * pos));
                const uint32_t sk = (psd_skip_bytes(x) >> (8 * pos + 7)) & 1u, ba = (psd_base_bytes(x) >> (8 * pos + 7)) & 1u;
                CHECK(sk == (ref_class(b) == 5), "skip mask of byte %u at %d in %08x", b, pos, x);
                CHECK(ba == (ref_class(b) < 4), "base mask of byte %u at %d in %08x", b, pos, x);
            }
    }
    for (uint32_t k = 0; k < 16; k++)
        for (int rep = 0; rep < 16; rep++) {
            const uint32_t v = rnd();
            uint32_t want = 0, j = 0;
            for (int i = 0; i < 4; i++)
                if ((k >> i) & 1u) want |= ((v >> (8 * i)) & 0xFFu) << (8 * j++);
            CHECK(psd_compact(v, k) == want, "psd_compact(%08x, %u)", v, k);
        }
}

// one chunk from incoming state s over [jlo, jhi): the word step's strings and the count summary
static void check_chunk(const uint8_t *p, int jlo, int jhi, uint32_t s, const char *what) {
    uint32_t w[16];
    load_words(p, w);
    std::vector<uint8_t> codes;
    const uint32_t s_end = ref_run(p, jlo, jhi, s, &codes);
    PsdBits o = {0, 0, 0, 0, s};
    psd_fasta_chunk(w, jlo, jhi, o);
    uint64_t hi = 0, lo = 0, bd = 0;
    for (size_t i = 0; i < codes.size(); i++) {
        hi = (hi << 2) | (lo >> 62);
        lo = (lo << 2) | (codes[i] & 3u);
        bd |= (uint64_t)(codes[i] >> 2) << i;
    }
    CHECK(o.n == codes.size() && o.s == s_end && o.sq_hi == hi && o.sq_lo == lo && o.bd == bd,
          "%s: chunk [%d, %d) from state %u: n %u/%zu state %u/%u", what, jlo, jhi, s, o.n, codes.size(), o.s, s_end);
    if (s == 0) {
        std::vector<uint8_t> c1;
        const uint32_t h_end = ref_run(p, jlo, jhi, 1, &c1);
        const uint32_t want_next = s_end | (h_end << 2) | (2u << 4) | (3u << 6);
        const uint64_t want_cnt = (uint64_t)codes.size() | ((uint64_t)c1.size() << 16);
        uint32_t next = 0;
        uint64_t cnt = 0;
        psd_fasta_count_bytes(w, jlo, jhi, next, cnt);
        CHECK(next == want_next && cnt == want_cnt, "%s: byte-wise count summary of [%d, %d): next %02x/%02x cnt %llx/%llx", what,
              jlo, jhi, next, want_next, (unsigned long long)cnt, (unsigned long long)want_cnt);
        bool has_gt = false;
        for (int i = 0; i < 64; i++) has_gt |= p[i] == '>';
        if (jlo == 0 && jhi == 64) {
            next = 0; cnt = 0;
            const bool took = psd_fasta_count_words(w, next, cnt);
            CHECK(took == !has_gt, "%s: word-wise count %s a chunk %s '>'", what, took ? "took" : "refused", has_gt ? "with" : "without");
            CHECK(!took || (next == want_next && cnt == want_cnt), "%s: word-wise count summary: next %02x/%02x cnt %llx/%llx", what,
                  next, want_next, (unsigned long long)cnt, (unsigned long long)want_cnt);
        }
    }
}

static const char ODD[] = {'N', 'n', 'R', 'y', 'W', '-', '*', ' ', '.', '\r', '\t', '\v', 0, 1, 31, 32, '@', '[', '`', '{',
                           (char)0x80, (char)0xC1, (char)0xD4, (char)0xFF, 'E', 'e', 'V', 'v', 'B', 'Q', 'q'};

static uint8_t rand_byte(int flavour) {
    const uint32_t r = rnd() % 100;
    if (r < 6) return '\n';
    if (flavour >= 1 && r < 9) return '>';
    if (flavour >= 2 && r < 25) return (uint8_t)ODD[rnd() % sizeof(ODD)];
    return (uint8_t)"ACGTacgtUu"[rnd() % (flavour >= 2 ? 10 : 4)];
}

// every [jlo, jhi) edge and both incoming states on random chunks, and a '>' at every byte
static void check_chunks() {
    uint8_t p[64];
    for (int trial = 0; trial < 240; trial++) {
        const int flavour = trial % 3;
        for (int i = 0; i < 64; i++) p[i] = rand_byte(flavour);
        for (int jlo = 0; jlo <= 64; jlo++)
            for (int jhi = jlo; jhi <= 64; jhi++)
                for (uint32_t s = 0; s < 2; s++) check_chunk(p, jlo, jhi, s, "random chunk");
    }
    for (int g = 0; g < 64; g++)
        for (int nl = -1; nl < 64; nl++) {
            for (int i = 0; i < 64; i++) p[i] = (uint8_t)"ACGT"[rnd() & 3];
            if (nl >= 0) p[nl] = '\n';
            p[g] = '>';
            for (uint32_t s = 0; s < 2; s++) {
                check_chunk(p, 0, 64, s, "'>' in a chunk of bases");
                check_chunk(p, g, 64, s, "'>' at the chunk's first byte");
                check_chunk(p, 0, g, s, "'>' just past the chunk's end");
            }
        }
}

// FASTA text of one line width: headers (some longer than two or three chunks), optional CRLF and lower case
static std::string make_fasta(int width, bool crlf, bool lower, int odd_per_mille, size_t len) {
    std::string t;
    int contig = 0;
    while (t.size() < len) {
        t += '>';
        const int hlen = (contig % 4 == 1) ? 100 + (int)(rnd() % 100) : (int)(rnd() % 20);
        for (int i = 0; i < hlen; i++) t += (char)('a' + rnd() % 26);
        t += crlf ? "\r\n" : "\n";
        const int body = 1 + (int)(rnd() % 3000);
        for (int i = 0; i < body; i++) {
            char c = "ACGT"[rnd() & 3];
            if (lower && (rnd() & 1)) c = (char)(c | 0x20);
            if ((int)(rnd() % 1000) < odd_per_mille) c = ODD[rnd() % sizeof(ODD)];
            t += c;
            if ((i + 1) % width == 0 || i + 1 == body) t += crlf ? "\r\n" : "\n";
        }
        contig++;
    }
    t.resize(len);
    return t;
}

// the whole text chunk by chunk, placed at output offset `lead`, against the reference reader + packing; and
// every chunk's count summary
static void check_stream(const std::string &text, size_t start, uint32_t lead, const char *what) {
    const uint8_t *t = (const uint8_t *)text.data();
    const size_t len = text.size();
    std::vector<uint8_t> codes;
    ref_run(t, (int)start, (int)len, 0, &codes);
    const size_t npos = lead + codes.size();
    std::vector<uint32_t> rseq(npos / 16 + 8, 0), rbad(npos / 32 + 8, 0);
    for (size_t i = 0; i < codes.size(); i++) {
        const size_t p = lead + i;
        rseq[p >> 4] |= (uint32_t)(codes[i] & 3) << (30 - 2 * (p & 15));
        rbad[p >> 5] |= (uint32_t)(codes[i] >> 2) << (p & 31);
    }
    std::vector<uint32_t> nseq(rseq.size(), 0), nbad(rbad.size(), 0);
    uint32_t state = 0;
    size_t pos = lead;
    for (size_t base = 0; base < len; base += 64) {
        uint8_t buf[64];
        memset(buf, 0, 64);
        memcpy(buf, t + base, len - base < 64 ? len - base : 64);
        const int jlo = start > base ? (int)(start - base < 64 ? start - base : 64) : 0;
        const int jhi = (int)(len - base < 64 ? len - base : 64);
        check_chunk(buf, jlo, jhi, 0, what);
        uint32_t w[16];
        load_words(buf, w);
        PsdBits o = {0, 0, 0, 0, state};
        psd_fasta_chunk(w, jlo, jhi, o);
        psd_place(o, (uint32_t)pos, nseq.data(), nbad.data(), [](uint32_t *p, uint32_t v) { *p |= v; });
        pos += o.n;
        state = o.s;
    }
    CHECK(pos == npos && nseq == rseq && nbad == rbad, "%s: len %zu start %zu lead %u: positions %zu/%zu seq %s bad %s", what,
          len, start, lead, pos, npos, nseq == rseq ? "ok" : "DIFFER", nbad == rbad ? "ok" : "DIFFER");
}

int main() {
    check_masks();
    check_chunks();
    for (int width = 1; width <= 200; width++) {
        const bool crlf = width % 3 == 0, lower = width % 2 == 0;
        const std::string text = make_fasta(width, crlf, lower, width % 5 == 0 ? 20 : 0, 4000 + rnd() % 4000);
        check_stream(text, (size_t)(width % 7 == 0 ? rnd() % 50 : 0), (uint32_t)(width % 32), "line width");
    }
    for (int width : {60, 61, 70, 80})
        for (uint32_t lead = 0; lead < 32; lead++) {
            const std::string text = make_fasta(width, lead % 4 == 3, lead % 2 == 1, lead % 3 == 0 ? 5 : 0, 3000 + rnd() % 3000);
            check_stream(text, lead % 5 == 0 ? rnd() % 70 : 0, lead, "every lead");
        }
    printf("%s: %d failing checks\n", failures ? "FAIL" : "OK", failures);
    return failures ? 1 : 0;
}
