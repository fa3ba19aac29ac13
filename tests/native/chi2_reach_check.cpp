// Host check of ps_chi2_reach (phenotypeseeker_b200/csrc/ps_chi2_reach.h) against every 2x2 table: for margins
// n1, n0, a threshold and a sample filter, every table (a present with phenotype 1, c present with phenotype 0)
// whose n_with = a + c lies outside the returned [lo, hi] must fail the filter or the kernel's screen
// (total (ad - bc)^2 / (row1 row2 col1 col2) < 0.99 chi2_min, in the kernel's operation order) or give NaN; and lo
// and hi themselves must each have a table that reaches 0.98 chi2_min. Built and run by tests/test_chi2_walk.py.
#include <stdio.h>
#include <stdint.h>
#include <math.h>
#include <initializer_list>
#include "../../phenotypeseeker_b200/csrc/ps_chi2_reach.h"

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint32_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (uint32_t)(rng_state >> 11); }

static int failures = 0, cases = 0;
#define CHECK(cond, ...) do { if (!(cond)) { if (failures++ < 20) { fprintf(stderr, __VA_ARGS__); fputc('\n', stderr); } } } while (0)

// the kernel's screen value for table (a, c), operation for operation (chi2_sp_finish in ps_test.cuh)
static double screen(int n1, int n0, int ai, int ci) {
    const double a = ai, c = ci, b = (double)n1 - a, d = (double)n0 - c;
    const double w_pheno = a + b, wo_pheno = c + d, w_kmer = a + c, wo_kmer = b + d;
    const double total = w_pheno + wo_pheno, det = a * d - b * c;
    return total * det * det / ((w_pheno * wo_pheno) * (w_kmer * wo_kmer));
}

static void check(int n1, int n0, int min_s, int max_s, double thr) {
    cases++;
    int lo, hi;
    ps_chi2_reach(n1, n0, min_s, max_s, thr, &lo, &hi);
    const double cmin = ps_chi2_min(thr);
    bool lo_hit = false, hi_hit = false;
    for (int a = 0; a <= n1; a++)
        for (int c = 0; c <= n0; c++) {
            const int m = a + c;
            const double v = screen(n1, n0, a, c);
            const bool filtered = m < min_s || n1 + n0 - m < 2 || m > max_s;
            if (m >= lo && m <= hi) {
                CHECK(!filtered, "n1 %d n0 %d min %d max %d: m %d in [%d, %d] fails the filter", n1, n0, min_s, max_s, m, lo, hi);
                if (v >= 0.98 * cmin && m == lo) lo_hit = true;
                if (v >= 0.98 * cmin && m == hi) hi_hit = true;
            } else {
                // dropped: must fail the filter, the screen, or be NaN (a NaN p-value never passes)
                CHECK(filtered || isnan(v) || v < 0.99 * cmin,
                      "n1 %d n0 %d min %d max %d thr %g: table a %d c %d (m %d, screen %.17g, chi2_min %.17g) outside [%d, %d]",
                      n1, n0, min_s, max_s, thr, a, c, m, v, cmin, lo, hi);
            }
        }
    if (lo <= hi) CHECK(lo_hit && hi_hit, "n1 %d n0 %d thr %g: bounds [%d, %d] not tight", n1, n0, thr, lo, hi);
}

int main() {
    const double thrs[] = {2.0, 1.0, 0.5, 1e-2, 1e-4, 5.5e-10, 1e-12, 0.0};
    // small N: every margin split and every filter edge
    for (int N = 2; N <= 24; N++)
        for (int n1 = 0; n1 <= N; n1++)
            for (double thr : thrs) {
                check(n1, N - n1, 2, N - 2, thr);
                check(n1, N - n1, 0, N, thr);
                check(n1, N - n1, 3, N - 4, thr);
                check(n1, N - n1, N, N, thr);
            }
    // random margins, with NA samples (n1 + n0 < N: the caller passes the non-NA counts) and without
    for (int it = 0; it < 60; it++) {
        const int N = it < 20 ? 5000 : it < 40 ? 8190 : 2 + (int)(rnd() % 3000);
        const int nna = it % 2 ? (int)(rnd() % (N / 10 + 1)) : 0;
        const int n1 = (int)(rnd() % (N - nna + 1)), n0 = N - nna - n1;
        const double thr = thrs[it % 8] * (it % 3 == 0 ? 1.0 : 0.37);
        const int min_s = it % 4 == 0 ? 0 : 2 + (int)(rnd() % 50), max_s = it % 5 == 0 ? N : N - 2 - (int)(rnd() % 50);
        check(n1, n0, min_s, max_s, thr);
    }
    // balanced and lopsided columns at the flagship size and at the largest N the walk takes
    for (int N : {5000, 8190})
        for (int n1 : {1, 2, 41, N / 3, N / 2, N - 42, N - 1})
            for (double thr : {5.5e-10, 1e-12, 1e-2}) check(n1, N - n1, 2, N - 2, thr);
    if (failures) { printf("FAIL %d of %d cases\n", failures, cases); return 1; }
    printf("OK %d cases\n", cases);
    return 0;
}
