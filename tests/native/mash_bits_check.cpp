// Host driver for phenotypeseeker_b200/csrc/ps_mash_bits.h (tests/test_weights_device.py compares its output with
// phenotypeseeker_b200/weights.py). Reads whitespace-separated queries from stdin, one answer per line on stdout:
//   h <k> <seed> <forward 2-bit word>        -> canonical word and h1 of its text
//   d <s> <na> <a...> <nb> <b...>            -> shared << 16 | denom
//   s <n> <x...> (hex floats)                -> the row sum of neighbour joining (psm_sum_*), as a hex float
#include <cinttypes>
#include <cstdio>
#include <vector>

#include "../../phenotypeseeker_b200/csrc/ps_mash_bits.h"

int main() {
    char op[4];
    while (scanf("%3s", op) == 1) {
        if (op[0] == 'h') {
            int k;
            uint32_t seed;
            uint64_t fw;
            if (scanf("%d %" SCNu32 " %" SCNu64, &k, &seed, &fw) != 3) return 2;
            const uint64_t canon = psm_canonical(fw, k);
            printf("%" PRIu64 " %" PRIu64 "\n", canon, psm_hash_kmer(canon, k, seed));
        } else if (op[0] == 'd') {
            uint32_t s, na, nb;
            if (scanf("%" SCNu32 " %" SCNu32, &s, &na) != 2) return 2;
            std::vector<uint64_t> a(na + 1), b;
            for (uint32_t i = 0; i < na; i++) if (scanf("%" SCNu64, &a[i]) != 1) return 2;
            if (scanf("%" SCNu32, &nb) != 1) return 2;
            b.resize(nb + 1);
            for (uint32_t i = 0; i < nb; i++) if (scanf("%" SCNu64, &b[i]) != 1) return 2;
            printf("%" PRIu32 "\n", psm_shared_denom(a.data(), na, b.data(), nb, s));
        } else if (op[0] == 's') {
            int n;
            if (scanf("%d", &n) != 1 || n < 1) return 2;
            PsmSum sum;
            for (int i = 0; i < n; i++) {
                double x;
                if (scanf("%la", &x) != 1) return 2;
                if (i == 0) psm_sum_first(sum, x);
                else psm_sum_add(sum, x);
            }
            printf("%a\n", psm_sum_end(sum));
        } else {
            return 2;
        }
    }
    return 0;
}
