// ps_chi2_reach.h — which k-mer sample counts can reach the chi2 threshold of a binary phenotype column.
// Host code (ps_test_chi2) and the host check tests/native/chi2_reach_check.cpp include it; no CUDA.
//
// For a column with n1 phenotype-1 and n0 phenotype-0 samples and a k-mer present in m of them, the 2x2 table
// is fixed by a = present & phenotype 1, a in [max(0, m - n0), min(m, n1)], and
//   chi2 = T (ad - bc)^2 / (n1 n0 m (T - m)),   T = n1 + n0,   ad - bc = a T - n1 m,
// a convex quadratic in a: its largest value over the tables is at one of the two ends of that interval.
// A margin of zero makes it 0/0 (NaN); the kernel's reference-order statistic is NaN then, and a NaN p-value
// never passes, so such a count is never reachable.
#pragma once
#include <math.h>

// p = exp(-chi2 / 2) < thr  <=>  chi2 > -2 ln thr: the bound the test kernels use (thr <= 0: nothing passes)
static inline double ps_chi2_min(double thr) { return thr > 0.0 ? -2.0 * log(thr) : 1e300; }

// largest chi2 over the tables with margins n1, n0 and n_with = m (NaN when a margin is zero)
static inline double ps_chi2_max_at(int n1, int n0, int m) {
    const double T = (double)n1 + (double)n0;
    const int alo = m - n0 > 0 ? m - n0 : 0, ahi = m < n1 ? m : n1;
    const double den = ((double)n1 * (double)n0) * ((double)m * (T - (double)m));
    const double d0 = (double)alo * T - (double)n1 * m, d1 = (double)ahi * T - (double)n1 * m;
    const double x0 = T * d0 * d0 / den, x1 = T * d1 * d1 / den;
    return x0 > x1 ? x0 : x1;    // both NaN or neither
}

// [*lo, *hi]: the smallest and largest n_with in [min_s, max_s] that passes the sample filter (n_with >= 0,
// n_without = n1 + n0 - n_with >= 2) and whose largest chi2 reaches 0.98 chi2_min. Every count is scanned: the
// reachable counts need not be contiguous, only their hull is returned. *lo > *hi when there is none.
// The kernel's own screen drops a table below 0.99 chi2_min; the 2 % margin keeps this cut looser than that
// screen whatever the rounding of either side, so it removes only tables the screen would remove.
static inline void ps_chi2_reach(int n1, int n0, int min_s, int max_s, double thr, int *lo, int *hi) {
    const double need = 0.98 * ps_chi2_min(thr);
    const int m0 = min_s > 0 ? min_s : 0;
    const int m1 = max_s < n1 + n0 - 2 ? max_s : n1 + n0 - 2;
    *lo = 1; *hi = 0;
    for (int m = m0; m <= m1; m++) {
        if (!(ps_chi2_max_at(n1, n0, m) >= need)) continue;
        if (*lo > *hi) *lo = m;
        *hi = m;
    }
}
