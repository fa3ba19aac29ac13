// ps_test.cuh — fused per-k-mer association test + p-value filter over the bit matrix.
//
// Replaces phenotypes.get_kmers_tested / conduct_chi_squared_test / conduct_t_test and their
// helpers (modeling.py:677-858). One pass over the matrix serves all phenotype columns.
//
// Thread mapping: a row is `wq` uint4 (128-bit) loads; LPR = pow2 >= wq lanes (<= 32)
// cooperate on one row, so a warp covers 32/LPR consecutive rows per step and every load
// instruction of the warp touches one contiguous, 16-byte-aligned span. Per-row partial sums
// are combined with xor-shuffles inside the lane group; lane 0 of the group finishes the
// statistic in FP64 and appends survivors through one atomic counter.
//
// chi2 (binary phenotype): 2x2 table a,b,c,d = sum of weights over (pheno 1/0) x
// (present/absent), NA samples skipped; expected = row*col/total; chi2 = sum (o-e)^2/e in cell
// order a,b,c,d; scipy.stats.chisquare(..., ddof=1) on 4 cells => df = 2 => p = exp(-chi2/2)
// (modeling.py:782-792). Unweighted tables are exact integers, so chi2 is bit-identical to
// the reference; weighted sums are accumulated per 128-bit lane then tree-combined (<= few
// ulp from the reference's sequential `+=`).
//
// Welch (continuous phenotype): statsmodels ttest_ind(usevar='unequal', weights=...) restated
// (SURVEY.md 8c): n_i = sum of weights, m_i weighted mean, v_i = sum w (x-m_i)^2 / n_i,
// sem_i = v_i/(n_i-1), t = (m1-m2)/sqrt(sem1+sem2), Satterthwaite dof,
// p = 2*t.sf(|t|, dof) = I_{dof/(dof+t^2)}(dof/2, 1/2) (regularised incomplete beta, FP64
// continued fraction).
#pragma once
#include <type_traits>
#include "ps_common.cuh"

struct SurvOut {
    int32_t *ph;
    unsigned long long *row;
    double *stat, *p, *mx, *my;
    uint32_t *n_with;
    unsigned long long *counter;
    unsigned long long cap;
};

__device__ __forceinline__ void surv_push(const SurvOut &o, int ph, unsigned long long row, double stat,
                                          double p, double mx, double my, uint32_t n_with) {
    const unsigned long long slot = atomicAdd(o.counter, 1ull);
    if (slot < o.cap) {
        o.ph[slot] = ph; o.row[slot] = row; o.stat[slot] = stat; o.p[slot] = p;
        o.mx[slot] = mx; o.my[slot] = my; o.n_with[slot] = n_with;
    }
}

// The min-p epilogue (ps_minp_*, permutation thresholds): the test kernels are instantiated with this in place of
// SurvOut. Nothing is compacted; every (row, column) pair that passes the sample filter and has a p (not NaN)
// offers it to minp[column], the bit pattern of the smallest p so far (1.0 before the pass). p >= 0, so the
// IEEE pattern orders like the value and one integer atomicMin keeps the minimum.
struct MinpOut {
    unsigned long long *minp;
};

template <class Out>
__device__ __forceinline__ constexpr bool is_minp() { return std::is_same<Out, MinpOut>::value; }

// The lanes lane ^ step, lane ^ 2 step, ... ^ 16 hold the same column; their smallest candidate goes to memory with
// one atomicMin from the owner lane, and only when it is below the value read there (a stale read is higher, never
// lower, so no minimum is lost). Called by all 32 lanes; cand = 1.0 offers nothing.
__device__ __forceinline__ void minp_offer(const MinpOut &o, int ph, bool owner, double cand, int step) {
    if (!__any_sync(0xffffffffu, cand < 1.0)) return;
    unsigned long long b = (unsigned long long)__double_as_longlong(cand);
    for (int s = step; s < 32; s <<= 1) b = min(b, __shfl_xor_sync(0xffffffffu, b, s));
    if (owner && b < __ldcg(o.minp + ph)) atomicMin(o.minp + ph, b);
}

__device__ __forceinline__ uint32_t u4_get(const uint4 &v, int j) {
    return j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w;
}

// ---------------------------------------------------------------------------------------
// chi-square. masks: [P][2][wp] words (pheno==1, pheno==0). totw: [P][2] = total weight of
// pheno==1 / pheno==0 samples. totn: [P] = number of non-NA samples. wtot: [P][2][wp] = total
// weight of the pheno==1 / pheno==0 samples of each 32-sample word.
//
// A row group (LPR lanes) first reduces the integer counts of up to LPR columns — every lane ends up
// with every sum — and lane j of the group keeps column j; then all lanes finish THEIR column at the
// same time (sample filter, one-division screen, reference-order chi2 in FP64). With 5,000 samples a
// row occupies a whole warp and ten columns are finished by ten lanes in parallel instead of one after
// the other on lane 0. Column masks are staged in shared memory (smem_masks != 0); a column without NA
// samples needs one popcount per word instead of two (absent-with-phenotype = popcount(row) - present).
// Out = SurvOut compacts the survivors (p < thr); Out = MinpOut keeps each column's smallest p (ps_minp_chi2).
template <bool WEIGHTED, int QPL, class Out = SurvOut>
__global__ void __launch_bounds__(256)
k_test_chi2(const uint4 *__restrict__ matrix, unsigned long long U, int wq, int lpr_log2, int P, int n_samples,
            const uint32_t *__restrict__ masks, const double *__restrict__ totw,
            const int *__restrict__ totn, const double *__restrict__ weights,
            const double *__restrict__ wtot, int min_s, int max_s, double thr, int smem_masks, Out out) {
    extern __shared__ uint32_t s_masks[];
    const int lpr = 1 << lpr_log2;
    const unsigned lane = threadIdx.x & 31;
    const unsigned sub = lane & (lpr - 1);
    const unsigned rpw = 32 >> lpr_log2;  // rows per warp step
    const unsigned long long warp_g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    const int wp = wq * 4;
    if (smem_masks) {
        for (int i = threadIdx.x; i < P * 2 * wp; i += blockDim.x) s_masks[i] = masks[i];
        __syncthreads();
    }
    const uint32_t *mbase = smem_masks ? s_masks : masks;
    // p = exp(-chi2/2) < thr  <=>  chi2 > -2 ln thr (thr <= 0: nothing can pass, any finite bound works)
    const double chi2_min = thr > 0.0 ? -2.0 * log(thr) : 1e300;
    for (unsigned long long r0 = warp_g * rpw; r0 < U; r0 += nwarps * rpw) {
        const unsigned long long r = r0 + (lane >> lpr_log2);
        const bool rvalid = r < U;
        uint4 rw[QPL];
#pragma unroll
        for (int q = 0; q < QPL; q++) {
            const int qi = sub + q * lpr;
            rw[q] = (rvalid && qi < wq) ? __ldg(matrix + r * (unsigned long long)wq + qi) : make_uint4(0, 0, 0, 0);
        }
        // A k-mer seen in fewer than min_s samples fails the sample filter of every column (n_with <= its
        // popcount): most union k-mers are private to one sample, so whole warps of rows stop here.
        uint32_t np = 0;
#pragma unroll
        for (int q = 0; q < QPL; q++) np += __popc(rw[q].x) + __popc(rw[q].y) + __popc(rw[q].z) + __popc(rw[q].w);
        for (int o = lpr >> 1; o > 0; o >>= 1) np += __shfl_xor_sync(0xffffffffu, np, o);
        if (__all_sync(0xffffffffu, !rvalid || (int)np < min_s)) continue;
        for (int p0 = 0; p0 < P; p0 += lpr) {
            uint32_t my_ai = 0, my_ci = 0;
            double my_a = 0.0, my_c = 0.0;
            for (int j = 0; j < lpr && p0 + j < P; j++) {
                const int ph = p0 + j;
                const uint32_t *m1 = mbase + (size_t)(ph * 2) * wp, *m0 = m1 + wp;
                const bool no_na = totn[ph] == n_samples;
                // exact integer part: present & pheno==1 / present & pheno==0
                uint32_t ai = 0, ci = 0;
#pragma unroll
                for (int q = 0; q < QPL; q++) {
                    const int qi = sub + q * lpr;
                    if (qi < wq) {
#pragma unroll
                        for (int jj = 0; jj < 4; jj++) {
                            const uint32_t w = u4_get(rw[q], jj);
                            const int wi = qi * 4 + jj;
                            ai += __popc(w & m1[wi]);
                            if (!no_na) ci += __popc(w & m0[wi]);
                        }
                    }
                }
                for (int o = lpr >> 1; o > 0; o >>= 1) {
                    ai += __shfl_xor_sync(0xffffffffu, ai, o);
                    if (!no_na) ci += __shfl_xor_sync(0xffffffffu, ci, o);
                }
                if (no_na) ci = np - ai;
                double a = 0.0, c = 0.0;
                if (WEIGHTED) {
                    const uint32_t n_with = ai + ci;
                    const int n_without = totn[ph] - (int)n_with;
                    // min/max sample filter first (modeling.py:770-772): most rows stop here
                    const bool tested = rvalid && !((int)n_with < min_s || n_without < 2 || (int)n_with > max_s);
                    if (tested) {
                        // per word, walk whichever is smaller: the set bits, or the cleared bits
                        // (then subtract from the word's total weight, wtot)
                        const double *wt1 = wtot + (size_t)(ph * 2) * wp, *wt0 = wt1 + wp;
#pragma unroll
                        for (int q = 0; q < QPL; q++) {
                            const int qi = sub + q * lpr;
                            if (qi < wq) {
#pragma unroll
                                for (int jj = 0; jj < 4; jj++) {
                                    const uint32_t w = u4_get(rw[q], jj);
                                    const int wi = qi * 4 + jj;
                                    const uint32_t k1 = m1[wi], k0 = m0[wi];
                                    uint32_t x1 = w & k1, y1 = ~w & k1, x0 = w & k0, y0 = ~w & k0;
                                    const double *wb = weights + wi * 32;
                                    if (__popc(x1) <= __popc(y1)) {
                                        while (x1) { const int bb = __ffs(x1) - 1; x1 &= x1 - 1; a += __ldg(wb + bb); }
                                    } else {
                                        double t = 0.0;
                                        while (y1) { const int bb = __ffs(y1) - 1; y1 &= y1 - 1; t += __ldg(wb + bb); }
                                        a += __ldg(wt1 + wi) - t;
                                    }
                                    if (__popc(x0) <= __popc(y0)) {
                                        while (x0) { const int bb = __ffs(x0) - 1; x0 &= x0 - 1; c += __ldg(wb + bb); }
                                    } else {
                                        double t = 0.0;
                                        while (y0) { const int bb = __ffs(y0) - 1; y0 &= y0 - 1; t += __ldg(wb + bb); }
                                        c += __ldg(wt0 + wi) - t;
                                    }
                                }
                            }
                        }
                    }
                    for (int o = lpr >> 1; o > 0; o >>= 1) {
                        // fixed tree: lower lane + upper lane, same value in both partners
                        const double a2 = __shfl_xor_sync(0xffffffffu, a, o), c2 = __shfl_xor_sync(0xffffffffu, c, o);
                        a = (lane & o) ? a2 + a : a + a2;
                        c = (lane & o) ? c2 + c : c + c2;
                    }
                }
                if ((int)sub == j) { my_ai = ai; my_ci = ci; my_a = a; my_c = c; }
            }
            // every lane finishes its own column; a `continue` inside the do-while(0) leaves the finish only, so
            // that the min-p epilogue after it is reached by the whole warp
            const int ph = p0 + (int)sub;
            double cand = 1.0;
            do {
            if (ph >= P || !rvalid) continue;
            const uint32_t n_with = my_ai + my_ci;
            const int n_without = totn[ph] - (int)n_with;
            if ((int)n_with < min_s || n_without < 2 || (int)n_with > max_s) continue;
            const double a = WEIGHTED ? my_a : (double)my_ai, c = WEIGHTED ? my_c : (double)my_ci;
            const double b = totw[ph * 2] - a, d = totw[ph * 2 + 1] - c;
            const double w_pheno = a + b, wo_pheno = c + d, w_kmer = a + c, wo_kmer = b + d;
            const double total = w_pheno + wo_pheno;
            // Cheap screen before the reference-order arithmetic (8 FP64 divisions + exp): for a 2x2
            // table sum (o-e)^2/e == total (ad - bc)^2 / (row1 row2 col1 col2), one division. Only rows
            // within 1 % of the threshold chi2 (or with a zero margin: NaN / inf) take the exact path,
            // so the survivors and their statistics are exactly those of the full computation.
            {
                const double det = a * d - b * c;
                const double approx = total * det * det / ((w_pheno * wo_pheno) * (w_kmer * wo_kmer));
                if (approx < 0.99 * chi2_min) continue;
            }
            const double ea = (w_pheno * w_kmer) / total, eb = (w_pheno * wo_kmer) / total;
            const double ec = (wo_pheno * w_kmer) / total, ed = (wo_pheno * wo_kmer) / total;
            const double ta = (a - ea) * (a - ea) / ea, tb = (b - eb) * (b - eb) / eb;
            const double tc = (c - ec) * (c - ec) / ec, td = (d - ed) * (d - ed) / ed;
            const double chi2 = ((ta + tb) + tc) + td;
            const double p = exp(-0.5 * chi2);
            if constexpr (is_minp<Out>()) { if (p < cand) cand = p; }
            else if (p < thr) surv_push(out, ph, r, chi2, p, 0.0, 0.0, n_with);  // NaN compares false
            } while (0);
            // lanes sub, sub + lpr, ... hold column ph; lane sub of the first row group offers their minimum
            if constexpr (is_minp<Out>()) minp_offer(out, ph, (int)lane < lpr && ph < P, cand, lpr);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Unweighted chi-square by walking the bits of the row instead of masking it once per column.
//
// k-mer presence is U-shaped: most union k-mers occur in a handful of samples (SNP variants) or in nearly
// all of them (core genome), and the masked-popcount kernel above spends 16 shared-memory mask words and 8
// POPC per lane and COLUMN on every row whatever it holds (ncu, 5,000 samples x 10 columns: 1,011 warp
// instructions per row, 75 % issue-bound, 205 shared wavefronts per row). Here every lane walks the set
// bits of its own words — or the cleared ones when the row is more than half full — and adds one packed
// word per bit: e1[s] holds, for ten columns at a time, a 12-bit field per column that is 1 iff sample s
// has phenotype 1 in that column (e0: phenotype 0; not needed when no column has NA samples, because then
// c = popcount(row) - a). One 128-bit load and two 64-bit adds per bit serve ten columns; the fields are
// summed over the lane group, and lane j finishes column j exactly like k_test_chi2 does.
// The counts are the same integers, so chi2 is bit-identical. Cost ~ min(n_with, N - n_with) per row.
// Field width 12 bits: min(popcount, N - popcount) <= 4095, i.e. N <= 8190 (the host checks).
//
// Rows whose popcount lies outside [np_lo, np_hi] are not walked: no column can reach the threshold with
// them (the host's ps_chi2_reach, one interval per column, reach[ph]; np_hi allows for the column's NA samples).
#define CHI2_SP_COLS 10      // columns per walk: two u64 of five 12-bit fields

template <int K>
__device__ __forceinline__ uint32_t pick_reg(const uint32_t (&v)[K], int i) {   // v[i] without local memory
    uint32_t x = v[0];
#pragma unroll
    for (int k = 1; k < K; k++) x = i == k ? v[k] : x;
    return x;
}

// Lane j of the row group finishes column ph from its summed fields: fa = number of walked samples with phenotype
// 1 in that column, fb = with phenotype 0 (the walked samples are the cleared ones of a dense row). A count
// outside reach[ph] fails the sample filter or the screen below; from the counts on, the arithmetic is that of
// k_test_chi2 (unweighted), operation for operation. With MinpOut the p lowers cand instead of being pushed.
template <bool NO_NA, class Out>
__device__ __forceinline__ void chi2_sp_finish(int ph, unsigned long long r, uint32_t fa, uint32_t fb, uint32_t np,
                                               bool dense, const int *__restrict__ tot1, const int *__restrict__ tot0,
                                               const int2 *__restrict__ reach, double chi2_min, double thr,
                                               const Out &out, double &cand) {
    const uint32_t ai = dense ? (uint32_t)tot1[ph] - fa : fa;
    const uint32_t ci = NO_NA ? np - ai : dense ? (uint32_t)tot0[ph] - fb : fb;
    const uint32_t n_with = ai + ci;
    const int2 rc = reach[ph];
    if ((int)n_with < rc.x || (int)n_with > rc.y) return;
    const double a = (double)ai, c = (double)ci;
    const double b = (double)tot1[ph] - a, d = (double)tot0[ph] - c;
    const double w_pheno = a + b, wo_pheno = c + d, w_kmer = a + c, wo_kmer = b + d;
    const double total = w_pheno + wo_pheno;
    {
        const double det = a * d - b * c;
        const double approx = total * det * det / ((w_pheno * wo_pheno) * (w_kmer * wo_kmer));
        if (approx < 0.99 * chi2_min) return;
    }
    const double ea = (w_pheno * w_kmer) / total, eb = (w_pheno * wo_kmer) / total;
    const double ec = (wo_pheno * w_kmer) / total, ed = (wo_pheno * wo_kmer) / total;
    const double ta = (a - ea) * (a - ea) / ea, tb = (b - eb) * (b - eb) / eb;
    const double tc = (c - ec) * (c - ec) / ec, td = (d - ed) * (d - ed) / ed;
    const double chi2 = ((ta + tb) + tc) + td;
    const double p = exp(-0.5 * chi2);
    if constexpr (is_minp<Out>()) { if (p < cand) cand = p; }
    else if (p < thr) surv_push(out, ph, r, chi2, p, 0.0, 0.0, n_with);  // NaN compares false
}

// Rows of at most 16 uint4 (N <= 2,048): LPR = pow2 >= wq lanes per row, one uint4 per lane, fields summed with
// xor-shuffles inside the group.
template <bool NO_NA, class Out = SurvOut>
__global__ void __launch_bounds__(256, 3)
k_test_chi2_sp(const uint4 *__restrict__ matrix, unsigned long long U, int wq, int lpr_log2, int P, int n_samples,
               const ulonglong2 *__restrict__ e1, const ulonglong2 *__restrict__ e0, int npad,
               const int *__restrict__ tot1, const int *__restrict__ tot0, const int2 *__restrict__ reach,
               int np_lo, int np_hi, double thr, Out out) {
    const int lpr = 1 << lpr_log2;
    const unsigned lane = threadIdx.x & 31;
    const unsigned sub = lane & (lpr - 1);
    const unsigned rpw = 32 >> lpr_log2;
    const unsigned long long warp_g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    const double chi2_min = thr > 0.0 ? -2.0 * log(thr) : 1e300;
    // the row of the NEXT step is loaded before this step's row is walked (the walk is short and would
    // otherwise wait out the whole DRAM latency of its own load: 26 % of the stall samples)
    auto load_row = [&](unsigned long long rr) {
        return (rr < U && (int)sub < wq) ? __ldg(matrix + rr * (unsigned long long)wq + sub) : make_uint4(0, 0, 0, 0);
    };
    uint4 nxt = load_row(warp_g * rpw + (lane >> lpr_log2));
    for (unsigned long long r0 = warp_g * rpw; r0 < U; r0 += nwarps * rpw) {
        const unsigned long long r = r0 + (lane >> lpr_log2);
        const bool rvalid = r < U;
        const uint4 rw = nxt;
        nxt = load_row(r + nwarps * rpw);
        uint32_t np = __popc(rw.x) + __popc(rw.y) + __popc(rw.z) + __popc(rw.w);
        for (int o = lpr >> 1; o > 0; o >>= 1) np += __shfl_xor_sync(0xffffffffu, np, o);
        const bool live = rvalid && (int)np >= np_lo && (int)np <= np_hi;
        if (__all_sync(0xffffffffu, !live)) continue;
        const bool dense = 2u * np > (uint32_t)n_samples;      // walk the cleared bits of the valid samples instead
        for (int c0 = 0; c0 < P; c0 += CHI2_SP_COLS) {
            const ulonglong2 *t1 = e1 + (size_t)(c0 / CHI2_SP_COLS) * npad;
            const ulonglong2 *t0 = NO_NA ? nullptr : e0 + (size_t)(c0 / CHI2_SP_COLS) * npad;
            unsigned long long a0 = 0, a1 = 0, b0 = 0, b1 = 0;
            if (live && (int)sub < wq) {
#pragma unroll
                for (int jj = 0; jj < 4; jj++) {
                    const int s0 = ((int)sub * 4 + jj) * 32;
                    uint32_t bits = u4_get(rw, jj);
                    if (dense) {
                        const int left = n_samples - s0;      // valid samples of this word
                        bits = ~bits & (left >= 32 ? 0xFFFFFFFFu : left <= 0 ? 0u : (1u << left) - 1u);
                    }
                    while (bits) {
                        const int s = s0 + __ffs(bits) - 1;
                        bits &= bits - 1;
                        const ulonglong2 v = __ldg(t1 + s);
                        a0 += v.x; a1 += v.y;
                        if (!NO_NA) { const ulonglong2 z = __ldg(t0 + s); b0 += z.x; b1 += z.y; }
                    }
                }
            }
            for (int o = lpr >> 1; o > 0; o >>= 1) {
                a0 += __shfl_xor_sync(0xffffffffu, a0, o);
                a1 += __shfl_xor_sync(0xffffffffu, a1, o);
                if (!NO_NA) { b0 += __shfl_xor_sync(0xffffffffu, b0, o); b1 += __shfl_xor_sync(0xffffffffu, b1, o); }
            }
            // lane j of the group finishes columns c0 + j, c0 + j + lpr, ... (min-p: in steps the whole warp takes,
            // each followed by the offer of the lanes that hold the same column)
            if constexpr (is_minp<Out>()) {
                for (int j0 = 0; j0 < CHI2_SP_COLS; j0 += lpr) {
                    const int j = j0 + (int)sub;
                    const bool mine = j < CHI2_SP_COLS && c0 + j < P;
                    double cand = 1.0;
                    if (live && mine) {
                        const int sh = 12 * (j % 5);
                        const uint32_t fa = (uint32_t)(((j < 5 ? a0 : a1) >> sh) & 4095ull);
                        const uint32_t fb = NO_NA ? 0u : (uint32_t)(((j < 5 ? b0 : b1) >> sh) & 4095ull);
                        chi2_sp_finish<NO_NA>(c0 + j, r, fa, fb, np, dense, tot1, tot0, reach, chi2_min, thr, out, cand);
                    }
                    minp_offer(out, c0 + j, (int)lane < lpr && mine, cand, lpr);
                }
                continue;
            }
            if (!live) continue;
            double unused = 1.0;
            for (int j = (int)sub; j < CHI2_SP_COLS && c0 + j < P; j += lpr) {
                const int sh = 12 * (j % 5);
                const uint32_t fa = (uint32_t)(((j < 5 ? a0 : a1) >> sh) & 4095ull);
                const uint32_t fb = NO_NA ? 0u : (uint32_t)(((j < 5 ? b0 : b1) >> sh) & 4095ull);
                chi2_sp_finish<NO_NA>(c0 + j, r, fa, fb, np, dense, tot1, tot0, reach, chi2_min, thr, out, unused);
            }
        }
    }
}

// The ten 12-bit fields of (x0, x1) as five u32 of two 16-bit fields: field j in p[j / 2] at bit 16 (j % 2).
// A lane's own fields are at most 256 (its words' bits), the warp's sums at most 4,095: no field carries.
__device__ __forceinline__ void fields16(unsigned long long x0, unsigned long long x1, uint32_t (&p)[5]) {
    const auto two = [](uint32_t v) { return (v & 0xFFFu) | ((v << 4) & 0xFFF0000u); };
    p[0] = two((uint32_t)x0);
    p[1] = two((uint32_t)(x0 >> 24));
    p[2] = (uint32_t)(x0 >> 48) | (((uint32_t)x1 & 0xFFFu) << 16);
    p[3] = two((uint32_t)(x1 >> 12));
    p[4] = two((uint32_t)(x1 >> 36));
#pragma unroll
    for (int i = 0; i < 5; i++) p[i] = __reduce_add_sync(0xffffffffu, p[i]);
}

// Rows that fill the warp (N > 2,048): lane l owns the 32-bit words l, l + 32, ... of the row, KW =
// ceil(W / 32) of them for the W words that hold samples, so no lane has more than one word more than another
// and each warp load is one 128-byte line. A lane walks all bits of all its words in ONE loop — when the current
// word is empty it takes the next non-empty one — so the warp runs max over lanes of the lane's bit count, not
// the sum over words of the per-word maxima. The fields are summed over the warp by REDUX (five u32 of two 16-bit
// fields) instead of twenty shuffles and adds; every lane gets every sum and lane j finishes column c0 + j.
template <int KW, bool NO_NA, class Out = SurvOut>
__global__ void __launch_bounds__(256, 3)
k_test_chi2_sp_warp(const uint32_t *__restrict__ matrix, unsigned long long U, int wp, int P, int n_samples,
                    const ulonglong2 *__restrict__ e1, const ulonglong2 *__restrict__ e0, int npad,
                    const int *__restrict__ tot1, const int *__restrict__ tot0, const int2 *__restrict__ reach,
                    int np_lo, int np_hi, double thr, Out out) {
    __shared__ uint32_t s_valid[KW * 32];    // s_valid[wi]: the bits of row word wi that are samples
    const int lane = (int)(threadIdx.x & 31);
    const int wv = (n_samples + 31) >> 5;
    for (int wi = threadIdx.x; wi < KW * 32; wi += blockDim.x) {
        const int left = n_samples - wi * 32;
        s_valid[wi] = left >= 32 ? 0xFFFFFFFFu : left <= 0 ? 0u : (1u << left) - 1u;
    }
    __syncthreads();
    const unsigned long long warp_g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    const double chi2_min = thr > 0.0 ? -2.0 * log(thr) : 1e300;
    // the next row is loaded before this one is walked, as in k_test_chi2_sp
    auto load_row = [&](unsigned long long rr, uint32_t (&dst)[KW]) {
#pragma unroll
        for (int k = 0; k < KW; k++) {
            const int wi = lane + 32 * k;
            dst[k] = (rr < U && wi < wv) ? __ldg(matrix + rr * (unsigned long long)wp + wi) : 0u;
        }
    };
    uint32_t nxt[KW];
    load_row(warp_g, nxt);
    for (unsigned long long r = warp_g; r < U; r += nwarps) {
        uint32_t w[KW];
#pragma unroll
        for (int k = 0; k < KW; k++) w[k] = nxt[k];
        load_row(r + nwarps, nxt);
        uint32_t np = 0;
#pragma unroll
        for (int k = 0; k < KW; k++) np += __popc(w[k]);
        np = __reduce_add_sync(0xffffffffu, np);
        if ((int)np < np_lo || (int)np > np_hi) continue;
        const bool dense = 2u * np > (uint32_t)n_samples;      // walk the cleared bits of the valid samples instead
        if (dense) {
#pragma unroll
            for (int k = 0; k < KW; k++) w[k] = ~w[k] & s_valid[lane + 32 * k];
        }
        uint32_t nz = 0;                                         // bit k: word k has bits to walk
#pragma unroll
        for (int k = 0; k < KW; k++) nz |= (w[k] != 0u ? 1u : 0u) << k;
        for (int c0 = 0; c0 < P; c0 += CHI2_SP_COLS) {
            const ulonglong2 *t1 = e1 + (size_t)(c0 / CHI2_SP_COLS) * npad;
            const ulonglong2 *t0 = NO_NA ? nullptr : e0 + (size_t)(c0 / CHI2_SP_COLS) * npad;
            unsigned long long a0 = 0, a1 = 0, b0 = 0, b1 = 0;
            uint32_t cur = 0, more = nz;
            int s0 = 0;
            while (cur | more) {
                if (cur == 0u) {
                    const int k = __ffs(more) - 1;
                    more &= more - 1u;
                    cur = pick_reg(w, k);
                    s0 = (lane + 32 * k) * 32;
                }
                const int s = s0 + __ffs(cur) - 1;
                cur &= cur - 1u;
                const ulonglong2 v = __ldg(t1 + s);
                a0 += v.x; a1 += v.y;
                if (!NO_NA) { const ulonglong2 z = __ldg(t0 + s); b0 += z.x; b1 += z.y; }
            }
            uint32_t fa[5], fb[5];
            fields16(a0, a1, fa);
            if (!NO_NA) fields16(b0, b1, fb);
            const bool mine = lane < CHI2_SP_COLS && c0 + lane < P;
            double cand = 1.0;
            if (mine) {
                const int sh = 16 * (lane & 1);
                const uint32_t ca = (pick_reg(fa, lane >> 1) >> sh) & 0xFFFFu;
                const uint32_t cb = NO_NA ? 0u : (pick_reg(fb, lane >> 1) >> sh) & 0xFFFFu;
                chi2_sp_finish<NO_NA>(c0 + lane, r, ca, cb, np, dense, tot1, tot0, reach, chi2_min, thr, out, cand);
            }
            // one row per warp: lane j alone holds column c0 + j
            if constexpr (is_minp<Out>()) minp_offer(out, c0 + lane, mine, cand, 32);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Regularised incomplete beta I_x(a, b), continued fraction (modified Lentz), FP64.
__device__ double ps_betacf(double a, double b, double x) {
    const double TINY = 1e-300, EPS = 1e-16;
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0, d = 1.0 - qab * x / qap;
    if (fabs(d) < TINY) d = TINY;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m <= 2000; m++) {
        const double m2 = 2.0 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d; if (fabs(d) < TINY) d = TINY;
        c = 1.0 + aa / c; if (fabs(c) < TINY) c = TINY;
        d = 1.0 / d;
        h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d; if (fabs(d) < TINY) d = TINY;
        c = 1.0 + aa / c; if (fabs(c) < TINY) c = TINY;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < EPS) break;
    }
    return h;
}

// two-sided Student-t p-value: 2*sf(|t|, dof) = I_{dof/(dof+t^2)}(dof/2, 1/2)
__device__ double ps_t_two_sided(double t, double dof) {
    if (isnan(t) || isnan(dof) || !(dof > 0.0)) return nan("");
    if (isinf(t)) return 0.0;
    if (isinf(dof)) return erfc(fabs(t) * 0.70710678118654752440);
    const double t2 = t * t;
    const double x = dof / (dof + t2);    // I_x(a, b)
    const double y = t2 / (dof + t2);     // 1 - x, no cancellation
    const double a = 0.5 * dof, b = 0.5;
    if (t2 == 0.0) return 1.0;
    const double lbt = lgamma(a + b) - lgamma(a) - lgamma(b) + a * log(x) + b * log(y);
    // far tail: fold the continued fraction into the exponent so the product does not
    // underflow before it has to (p stays exact down to the denormal range, like scipy)
    if (x < (a + 1.0) / (a + b + 2.0)) return exp(lbt + log(ps_betacf(a, b, x) / a));
    return 1.0 - exp(lbt) * ps_betacf(b, a, y) / b;
}

// Welch. nonna: [P][wp] words; vals: [P][N] phenotype values CENTRED on the weighted mean mu_p of the
// non-NA samples; weights: [N] (NULL = 1); tot: [P][4] = { sum w, sum w*vc, sum w*vc^2, mu_p } over
// the non-NA samples; totn: [P] = number of non-NA samples.
//
// Only the SMALLER of the two groups (with / without the k-mer) is walked bit by bit, twice (mean,
// then squared deviations: exact, also for a zero-variance group). The larger group follows from the
// centred totals by subtraction. If that leaves a variance that is zero within rounding while the
// small group's variance is exactly zero — the one case where the reference yields NaN and drops
// the k-mer — the larger group is recomputed directly by one lane (rare).
__device__ __forceinline__ void welch_direct_group(const uint32_t *__restrict__ rowp, const uint32_t *__restrict__ mk,
                                                   int wp, bool present, const double *__restrict__ pv,
                                                   const double *__restrict__ weights, double &sw, double &mean,
                                                   double &var) {
    double a = 0, b = 0;
    for (int wi = 0; wi < wp; wi++) {
        uint32_t g = (present ? rowp[wi] : ~rowp[wi]) & mk[wi];
        while (g) { const int s = wi * 32 + __ffs(g) - 1; g &= g - 1;
            const double ww = weights ? weights[s] : 1.0; a += ww; b += ww * pv[s]; }
    }
    sw = a; mean = b / a;
    double q = 0;
    for (int wi = 0; wi < wp; wi++) {
        uint32_t g = (present ? rowp[wi] : ~rowp[wi]) & mk[wi];
        while (g) { const int s = wi * 32 + __ffs(g) - 1; g &= g - 1;
            const double ww = weights ? weights[s] : 1.0; const double d = pv[s] - mean; q += ww * d * d; }
    }
    var = q / a;
}

template <int QPL, class Out = SurvOut>
__global__ void __launch_bounds__(256)
k_test_welch(const uint4 *__restrict__ matrix, unsigned long long U, int wq, int lpr_log2, int P, int N,
             const uint32_t *__restrict__ nonna, const double *__restrict__ vals,
             const double *__restrict__ weights, const double *__restrict__ tot, const int *__restrict__ totn,
             int min_s, int max_s, double thr, double t_min, Out out) {
    const int lpr = 1 << lpr_log2;
    const unsigned lane = threadIdx.x & 31;
    const unsigned sub = lane & (lpr - 1);
    const unsigned rpw = 32 >> lpr_log2;
    const unsigned long long warp_g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    const int wp = wq * 4;
    const int src0 = lane & ~(lpr - 1);  // lane 0 of my group
    for (unsigned long long r0 = warp_g * rpw; r0 < U; r0 += nwarps * rpw) {
        const unsigned long long r = r0 + (lane >> lpr_log2);
        const bool rvalid = r < U;
        uint4 rw[QPL];
#pragma unroll
        for (int q = 0; q < QPL; q++) {
            const int qi = sub + q * lpr;
            rw[q] = (rvalid && qi < wq) ? __ldg(matrix + r * (unsigned long long)wq + qi) : make_uint4(0, 0, 0, 0);
        }
        {   // fewer than min_s samples carry the k-mer: no column can test it (see k_test_chi2)
            uint32_t np = 0;
#pragma unroll
            for (int q = 0; q < QPL; q++) np += __popc(rw[q].x) + __popc(rw[q].y) + __popc(rw[q].z) + __popc(rw[q].w);
            for (int o = lpr >> 1; o > 0; o >>= 1) np += __shfl_xor_sync(0xffffffffu, np, o);
            if (__all_sync(0xffffffffu, !rvalid || (int)np < min_s)) continue;
        }
        for (int ph = 0; ph < P; ph++) {
            const uint32_t *mk = nonna + (size_t)ph * wp;
            const double *pv = vals + (size_t)ph * N;
            uint32_t nx = 0;
#pragma unroll
            for (int q = 0; q < QPL; q++) {
                const int qi = sub + q * lpr;
                if (qi < wq) {
#pragma unroll
                    for (int j = 0; j < 4; j++) nx += __popc(u4_get(rw[q], j) & __ldg(mk + qi * 4 + j));
                }
            }
            for (int o = lpr >> 1; o > 0; o >>= 1) nx += __shfl_xor_sync(0xffffffffu, nx, o);
            const uint32_t ny = (uint32_t)totn[ph] - nx;
            const bool tested = rvalid && !((int)nx < min_s || (int)ny < 2 || (int)nx > max_s);
            const bool small_x = nx <= ny;      // walk the group with the k-mer, or the one without
            // pass 1 over the small group: weight sum, weighted centred sum and sum of squares
            double sw = 0, sv = 0, sq = 0;
            if (tested) {
#pragma unroll
                for (int q = 0; q < QPL; q++) {
                    const int qi = sub + q * lpr;
                    if (qi < wq) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const int wi = qi * 4 + j;
                            const uint32_t w = u4_get(rw[q], j);
                            uint32_t g = (small_x ? w : ~w) & __ldg(mk + wi);
                            while (g) { const int s = wi * 32 + __ffs(g) - 1; g &= g - 1;
                                const double ww = weights ? __ldg(weights + s) : 1.0, v = __ldg(pv + s), wv = ww * v;
                                sw += ww; sv += wv; sq += wv * v; }
                        }
                    }
                }
            }
            for (int o = lpr >> 1; o > 0; o >>= 1) {
                sw += __shfl_xor_sync(0xffffffffu, sw, o);
                sv += __shfl_xor_sync(0xffffffffu, sv, o);
                sq += __shfl_xor_sync(0xffffffffu, sq, o);
            }
            sw = __shfl_sync(0xffffffffu, sw, src0);
            sv = __shfl_sync(0xffffffffu, sv, src0);
            sq = __shfl_sync(0xffffffffu, sq, src0);
            const double ms = sv / sw;           // centred mean of the small group
            // Sum of squared deviations from the moments of that one walk: sq - sv^2/sw. Its relative error is
            // ~2^-52 * sq / qs, so it stands whenever qs > 1e-8 sq (error < 1e-8, tolerance 1e-6); a group that is
            // constant or nearly so (qs tiny against sq: discrete phenotypes) is walked a second time, exactly.
            const double qs1 = sq - sv * ms;
            const bool exact2 = tested && !(qs1 > 1e-8 * sq);
            double qs = 0;
            if (exact2) {
#pragma unroll
                for (int q = 0; q < QPL; q++) {
                    const int qi = sub + q * lpr;
                    if (qi < wq) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const int wi = qi * 4 + j;
                            const uint32_t w = u4_get(rw[q], j);
                            uint32_t g = (small_x ? w : ~w) & __ldg(mk + wi);
                            while (g) { const int s = wi * 32 + __ffs(g) - 1; g &= g - 1;
                                const double ww = weights ? __ldg(weights + s) : 1.0; const double dv = __ldg(pv + s) - ms; qs += ww * dv * dv; }
                        }
                    }
                }
            }
            for (int o = lpr >> 1; o > 0; o >>= 1) qs += __shfl_xor_sync(0xffffffffu, qs, o);
            if (!exact2) qs = qs1;
            // lane 0 of each row group finishes the row; a `continue` inside the do-while(0) leaves the finish
            // only, so that the min-p epilogue after it is reached by the whole warp
            double cand = 1.0;
            do {
            if (sub != 0 || !tested) continue;
            const double Tw = tot[ph * 4], Twv = tot[ph * 4 + 1], Twvv = tot[ph * 4 + 2], mu = tot[ph * 4 + 3];
            const double var_s = qs / sw;
            double swL = Tw - sw, mL = (Twv - sv) / swL;
            double var_L = (Twvv - (qs + sw * ms * ms)) / swL - mL * mL;
            if (var_L < 0.0) var_L = 0.0;
            if (var_L <= 1e-9 * (Twvv / Tw)) {
                // the larger group is (nearly) constant: what the subtraction left is cancellation noise of the
                // centred totals, whatever the small group looks like — recompute it exactly, like the reference
                welch_direct_group(reinterpret_cast<const uint32_t *>(matrix) + r * (unsigned long long)wp, mk, wp,
                                   !small_x, pv, weights, swL, mL, var_L);
            }
            const double n1 = small_x ? sw : swL, n2 = small_x ? swL : sw;
            const double m1c = small_x ? ms : mL, m2c = small_x ? mL : ms;
            const double v1 = small_x ? var_s : var_L, v2 = small_x ? var_L : var_s;
            const double s1 = v1 / (n1 - 1.0), s2 = v2 / (n2 - 1.0);
            const double t = (m1c - m2c) / sqrt(s1 + s2);
            const double r1 = s1 / (s1 + s2), r2 = s2 / (s1 + s2);
            // Student's t has heavier tails than the normal at every dof: p >= erfc(|t| / sqrt 2). Below t_min
            // (the normal quantile of the threshold) p cannot pass, and the incomplete-beta evaluation (lgamma,
            // log, a continued fraction — thousands of FP64 operations on one lane) is skipped. NaN falls through.
            if (fabs(t) < t_min) continue;
            const double dof = 1.0 / (r1 * r1 / (n1 - 1.0) + r2 * r2 / (n2 - 1.0));
            const double p = ps_t_two_sided(t, dof);
            if constexpr (is_minp<Out>()) { if (p < cand) cand = p; }
            else if (p < thr) surv_push(out, ph, r, t, p, mu + m1c, mu + m2c, nx);
            } while (0);
            // lanes 0, lpr, 2 lpr, ... hold column ph for their rows; lane 0 offers the minimum
            if constexpr (is_minp<Out>()) minp_offer(out, ph, lane == 0, cand, lpr);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Top-k by p-value per phenotype column (the `--n_kmers` cut of get_ML_df, modeling.py:1128-1131, in
// numeric order): radix-select on the bit pattern of p (p >= 0, so the pattern orders like the value).
// One round = one byte, most significant first: histogram of that byte over the survivors whose higher
// bytes equal the phenotype's prefix; the host walks 256 counters per column to extend the prefix.
__global__ void k_sel_hist(const int32_t *__restrict__ ph, const double *__restrict__ p, unsigned long long ns,
                           const unsigned long long *__restrict__ prefix, int shift, uint32_t *__restrict__ hist) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < ns;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const int c = ph[i];
        const unsigned long long b = (unsigned long long)__double_as_longlong(p[i]);
        if (shift == 56 || (b >> (shift + 8)) == prefix[c]) atomicAdd(&hist[c * 256 + (int)((b >> shift) & 255ull)], 1u);
    }
}

// keeps survivor i iff bits(p) <= thr[column]; compacts the SoA into the `o` arrays
__global__ void k_sel_compact(SurvOut in, unsigned long long ns, const unsigned long long *__restrict__ thr, SurvOut o) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < ns;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const int c = in.ph[i];
        if ((unsigned long long)__double_as_longlong(in.p[i]) <= thr[c])
            surv_push(o, c, in.row[i], in.stat[i], in.p[i], in.mx[i], in.my[i], in.n_with[i]);
    }
}
