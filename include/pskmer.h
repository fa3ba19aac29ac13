/*
 * pskmer.h — C-ABI of libpskmer.so, the B200-native (sm_100a) replacement for the
 * data-parallel hot path of `phenotypeseeker modeling`.
 *
 * The reference (bioinfo-ut/PhenotypeSeeker v1.2.4) has no FFI: the path sits behind
 * subprocess calls to GenomeTester4 tools plus per-k-mer Python loops. Each entry point
 * below names the reference interface it replaces (file:line relative to the reference
 * root). INTEGRATION.md shows the ctypes stub a maintainer adds to modeling.py.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; ps_last_error() gives the text.
 *     Nothing here calls exit()/abort().
 *   - plain pointers and sizes only. Bulk input pointers may be host OR device
 *     pointers (unified virtual addressing decides); output pointers are host.
 *   - one ps_ctx per GPU, used from one host thread. The CUDA context is created by
 *     ps_ctx_create, never at library load (the reference forks Pools around the call).
 *   - sample order = row order of data.pheno = bit order in matrix rows:
 *     sample s is bit (s & 31) of word (s >> 5) of a row.
 *   - k-mers are 2 bits/base, A=0 C=1 G=2 T=3, first base most significant, canonical
 *     = min(word, reverse complement) — the GenomeTester4 .list encoding.
 */
#ifndef PSKMER_H
#define PSKMER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ps_ctx ps_ctx;

#define PS_OK 0
#define PS_ERR_ARG -1
#define PS_ERR_CUDA -2
#define PS_ERR_STATE -3
#define PS_ERR_NOMEM -4

int ps_version(void);

/* Create / destroy the per-GPU context (owns all device memory and one stream). */
int ps_ctx_create(int device, ps_ctx **out);
void ps_ctx_destroy(ps_ctx *ctx);
/* Last error text of ctx (or of ps_ctx_create when ctx == NULL). */
const char *ps_last_error(ps_ctx *ctx);

/*
 * Start a new job: k-mer length (1..32), number of samples (1..65535) and the
 * per-sample minimum count `cutoff` (>= 1; "-c", scripts/phenotypeseeker:93-96).
 * Drops all samples / union / results of the previous job but keeps device buffers.
 * Replaces: Input.Input_args plumbing of kmer_length / cutoff, modeling.py:161-162.
 */
int ps_begin(ps_ctx *ctx, int k, int n_samples, uint32_t cutoff);

/*
 * Restrict the job to canonical k-mers in [lo, hi) — the k-mer-space shard this GPU
 * owns (multi-GPU) or the partition being processed (memory-bounded runs).
 * Default after ps_begin: the whole space. (No reference equivalent; SURVEY.md §8e.)
 */
int ps_set_range(ps_ctx *ctx, uint64_t lo, uint64_t hi);

/*
 * Memory-bounded runs on one GPU, part 1: extract the instances of every k-mer in [lo, hi) (0, 0 = the whole
 * space) from all samples ONCE and leave them, partitioned by their top k-mer byte, in the level-1 page pool
 * (4 B per instance; n_instances = upper estimate for that range, 0 = every position of the input).
 * ps_set_range + ps_build_union calls that follow with sub-ranges of [lo, hi) whose inner boundaries are
 * multiples of 4^(k-4) (top-byte boundaries) start from that pool instead of walking the input again, so a
 * job cut into R k-mer ranges for lack of memory extracts its k-mers S < R times (S = pools of this size
 * that fit). k = 9..16. Any other range, a new sample or ps_begin drops the pool. (No reference equivalent;
 * SURVEY.md §7 "memory at config 5".)
 */
int ps_scatter_range(ps_ctx *ctx, uint64_t lo, uint64_t hi, uint64_t n_instances);

/*
 * Memory-bounded runs, part 0 (optional): announce, before the first ps_add_samples of a job, the k-mer range
 * [lo, hi) that ps_scatter_range will be asked for first and the capacity of its pool (n_instances, as there;
 * share = expected share of all instances that falls into the range, used for profile accounting only). Every
 * sample is then scattered for that range right after it has been decoded — for host input that is while the
 * next 64 MB of text are still crossing PCIe — and ps_scatter_range(lo, hi, ...) only closes the pages.
 * n_instances = 0 switches it off. cutoff 1, assemblies, k = 9..16; ignored otherwise.
 */
int ps_ingest_scatter(ps_ctx *ctx, uint64_t lo, uint64_t hi, uint64_t n_instances, double share);

/*
 * Memory hint for range-restricted builds: an upper estimate of the k-mer instances (positions) that
 * fall into the current range. The page pools of the next ps_build_union are sized from it instead of
 * from the whole input; if the range turns out to hold more, the build repeats itself with larger pools.
 * 0 (default after ps_begin) = size for every position of the input.
 */
int ps_set_capacity_hint(ps_ctx *ctx, uint64_t n_instances);

/*
 * Stage 1 — ingest `count` samples idx = first_idx .. first_idx+count-1 from raw
 * FASTA/FASTQ text (host or device pointers): decode to a 2-bit packed stream plus an
 * invalid-position bitmask on device. FASTQ samples, and all samples when cutoff > 1,
 * are also counted per sample (radix sort + run-length) with the cutoff applied.
 * Replaces: Samples.get_kmer_lists -> `glistmaker <fa> -o ... -w k -c c`,
 * modeling.py:303-315.
 */
int ps_add_samples(ps_ctx *ctx, int first_idx, int count,
                   const void *const *bytes, const size_t *lens);

/*
 * One sample's sorted distinct canonical k-mers with counts (count >= cutoff), i.e. the
 * content of `glistquery <sample>.list`. Two-call pattern: with kmers == NULL only *n
 * is set. Replaces: the .list file of glistmaker (modeling.py:309-310; Appendix A1).
 */
int ps_sample_kmers(ps_ctx *ctx, int idx, uint32_t cutoff,
                    uint64_t *kmers, uint32_t *counts, size_t cap, size_t *n);

/*
 * Stage 2 — union of all samples' k-mer sets (ascending) and the k-mer-major,
 * bit-packed presence matrix [U][row_words]. *n_union = U of this range.
 * Replaces: Samples.get_feature_vector/get_union (`glistcompare -u`, modeling.py:351-380),
 * Samples.map_samples (`glistquery -l`, `split`, :317-348) and
 * phenotypes.kmer_testing_setup's `wc -l` (:641-644).
 */
int ps_build_union(ps_ctx *ctx, uint64_t *n_union);

/* Row stride of the matrix in 32-bit words (ceil(N/32) rounded up to 4). */
int ps_row_words(ps_ctx *ctx);
/* Copy out union k-mers [first, first+count) and their matrix rows (parity / tests). */
int ps_get_union(ps_ctx *ctx, uint64_t first, uint64_t count, uint64_t *kmers);
int ps_get_rows(ps_ctx *ctx, uint64_t first, uint64_t count, uint32_t *rows);

/*
 * Install a union + matrix computed elsewhere (host or device pointers; kmers may be NULL):
 * U rows of ps_row_words() words. Lets stage 3 run on a stored matrix (the reference's
 * analogue is re-reading the K-mer_lists/*_mapped_* stripes, modeling.py:650-657) and lets
 * tests drive the test kernels with arbitrary presence vectors.
 */
int ps_load_matrix(ps_ctx *ctx, uint64_t n_union, const uint64_t *kmers, const uint32_t *rows);

/*
 * --kmerDB: cut the union down to the k-mers that also occur in `db_kmers` (n_db ascending distinct canonical
 * k-mers, host or device pointer — e.g. what ps_sample_kmers returned for the database FASTA) and keep their
 * matrix rows; both stay on the device. *n_union = size of the intersection, which is what
 * kmer_testing_setup then counts (modeling.py:641-644). Call after ps_build_union.
 * Replaces: `glistmaker <kmerDB>` + `glistcompare -i` + `mv` of Samples.get_feature_vector, modeling.py:367-372.
 */
int ps_restrict_union(ps_ctx *ctx, const uint64_t *db_kmers, size_t n_db, uint64_t *n_union);

/*
 * Stage 3 — fused per-k-mer test + p-value filter over the bit matrix, all `n_pheno`
 * phenotype columns in one pass. A (k-mer, column) pair survives iff the min/max
 * sample filter passes and p < p_threshold (the caller folds Bonferroni in:
 * pvalue_cutoff / U, or pvalue_cutoff with --omit_B_correction).
 *
 * chi2: pheno[p*N + s] in {1, 0, -1 = NA}; weights NULL = unweighted (exact integers).
 * Replaces: phenotypes.get_kmers_tested + conduct_chi_squared_test and helpers,
 * modeling.py:677-714, 759-858 (scipy.stats.chisquare ddof=1 -> p = exp(-chi2/2)).
 *
 * welch: pheno[p*N + s] double, NaN = NA. Weighted Welch t-test,
 * p = 2 * t.sf(|t|, dof_satterthwaite).
 * Replaces: conduct_t_test + statsmodels ttest_ind(usevar='unequal', weights=...),
 * modeling.py:716-757.
 */
int ps_test_chi2(ps_ctx *ctx, int n_pheno, const int8_t *pheno, const double *weights,
                 int min_samples, int max_samples, double p_threshold,
                 uint64_t *n_survivors);
int ps_test_welch(ps_ctx *ctx, int n_pheno, const double *pheno, const double *weights,
                  int min_samples, int max_samples, double p_threshold,
                  uint64_t *n_survivors);

/*
 * Permutation min-p: minp[c] = smallest p over the k-mers of this range's union that pass the sample filter,
 * for each of the n_cols phenotype columns given (1 if none). Leaves union, matrix and the survivors of the
 * last ps_test_* call untouched.
 *
 * Same table layout and conventions as ps_test_chi2 / ps_test_welch (column c at pheno[c*N + s]); the
 * columns are typically permutations of an observed column. The statistic and p of a (k-mer, column) pair
 * are those ps_test_* computes; a NaN p is never a minimum. Runs the columns in batches, one pass over the
 * matrix per batch. For Westfall & Young's single-step min-p threshold (DESIGN.md "Permutation threshold").
 */
int ps_minp_chi2(ps_ctx *ctx, int n_cols, const int8_t *pheno, const double *weights,
                 int min_samples, int max_samples, double *minp);
int ps_minp_welch(ps_ctx *ctx, int n_cols, const double *pheno, const double *weights,
                  int min_samples, int max_samples, double *minp);

/*
 * Top-k cut on device: of the survivors of the last ps_test_* call keep, for every phenotype column, the
 * n_top with the smallest p-values (numeric order; every survivor tied with the n_top-th is kept too, so
 * slightly more than n_top may remain). ps_fetch_survivors then returns only those. *n_selected = how
 * many remain over all columns.
 * Replaces: the `--n_kmers` cut of phenotypes.get_ML_df (sort by p-value, first kmer_limit columns),
 * modeling.py:1128-1131 — there on "%.2E" strings; callers that need that exact order fetch all survivors.
 */
int ps_select_top(ps_ctx *ctx, int n_pheno, uint64_t n_top, uint64_t *n_selected);

/*
 * Survivors of the last ps_test_* call, ordered by (pheno_idx, row). Any output
 * pointer may be NULL. rowbits: cap * ps_row_words() words. mean_x / mean_y are
 * filled by the Welch test only. row = rank of the k-mer in this range's union.
 * Replaces: the dict returned by get_kmers_tested / pheno.ML_df, modeling.py:670-672,
 * 739, 796.
 */
int ps_fetch_survivors(ps_ctx *ctx, size_t cap, int32_t *pheno_idx, uint64_t *row,
                       uint64_t *kmer, double *stat, double *p, double *mean_x,
                       double *mean_y, uint32_t *n_with, uint32_t *rowbits);

/*
 * Occurrence counts of K given canonical k-mers in sample idx (0 if absent): the
 * count == 1 case of ps_count_matrix, same rules.
 */
int ps_lookup(ps_ctx *ctx, int idx, const uint64_t *kmers, size_t K, uint32_t *counts);

/*
 * counts[i*K + j] = occurrences of kmers[j] in sample first_idx + i, for i < count:
 * one device pass over the decoded streams of all those samples.
 * kmers: K <= 2^30 canonical codes (host or device memory), duplicates allowed (every
 * copy gets the count). A count covers every valid window of the sample's decoded
 * stream: it is not cut by the job's cutoff or k-mer range. counts: host memory.
 * The job's union, matrix, survivors and k-mer range are left untouched.
 * PS_ERR_ARG for a sample that is not present, null pointers, or count x K overflow.
 * Replaces: `gmer_counter -db <kmers> <sample>` of prediction.py:72-100 for every
 * sample, and the raw-count columns of --real_counts (modeling.py:693-695).
 */
int ps_count_matrix(ps_ctx *ctx, int first_idx, int count, const uint64_t *kmers, size_t K,
                    uint32_t *counts);

/*
 * Packed streams for the multi-GPU exchange (device pointers, valid until ps_begin):
 * seq = 2 bits/base, 16 bases per u32, first base in the top bits; bad = 1 bit per
 * position (bit i&31 of word i>>5), 1 = window break. n_pos positions, padded to a
 * multiple of 4096 with bad positions. ps_import_stream copies device -> device.
 */
int ps_export_stream(ps_ctx *ctx, int idx, const void **seq, const void **bad, uint64_t *n_pos);
int ps_import_stream(ps_ctx *ctx, int idx, const void *seq, const void *bad, uint64_t n_pos);
/* Same for `count` consecutive samples whose streams lie back to back in seq / bad. */
int ps_import_streams(ps_ctx *ctx, int first_idx, int count, const void *seq, const void *bad,
                      const uint64_t *n_pos);
/*
 * Multi-GPU routing (the exchange step of SURVEY.md 8e) for k = 9..16. The k-mer space is cut into
 * nparts contiguous ranges by nparts - 1 ascending splitters; GPU d owns [splitters[d-1], splitters[d]).
 * Every GPU keeps a receive pool of pages (4 KB, 1024 four-byte records) cut into nparts sub-pools of
 * pages_per_sender pages, one per sending GPU, plus one meta word per page. The extraction kernel of
 * a sender groups its k-mer instances by (owner, top k-mer byte) and appends each group directly to
 * pages of the owner's pool — plain stores over NVLink when the pool is a peer's (CUDA IPC mapping),
 * so the all-to-all is the write-out of the extraction kernel. No counts are exchanged.
 *
 *   ps_route_pages_needed  sub-pool size this GPU needs in every receiver for the samples it holds when the
 *                          k-mer space is covered in `passes` passes; the job uses the maximum over all GPUs.
 *   ps_route_setup         sizes this GPU's pool; returns the device pointers to export (ps_ipc_export).
 *                          nparts == 0 ends routed mode.
 *   ps_route_peers         pools of all ranks (own pointers for my_rank, ps_ipc_open mappings for peers —
 *                          or plain device pointers of other contexts on the same GPU).
 *   ps_route_begin         clears this GPU's page metas; every rank must have done so (barrier) before
 *                          anybody scatters.
 *   ps_route_scatter       extraction + scatter of this GPU's samples into all pools (asynchronous on
 *                          ps_stream; the data is complete on the receivers once every rank's stream
 *                          has passed this call — barrier). With ps_set_range only k-mers of that
 *                          super-range travel (jobs too large for one pass: one pass per super-range,
 *                          the splitters of a pass lie inside its super-range).
 *   ps_route_build         union + matrix of this GPU's range from its pool, like ps_build_union.
 *                          *overflow = 1 if this GPU ran out of pages as a sender (results invalid:
 *                          repeat with larger pools; every rank should learn it with the U all-reduce).
 * Replaces: the N lists -> one feature vector -> N mapped stripes regrouping of modeling.py:317-380,
 * sharded over GPUs.
 */
int ps_route_pages_needed(ps_ctx *ctx, int nparts, int passes, uint64_t *pages);
/* Upper bound of the k-mer instances the samples held by this context contribute to a build (stream positions of
 * assemblies, distinct counted k-mers of raw-read / cutoff samples): what pool sizes and pass counts are planned from. */
uint64_t ps_instances_upper(ps_ctx *ctx);
int ps_route_setup(ps_ctx *ctx, int nparts, int my_rank, const uint64_t *splitters, uint64_t pages_per_sender,
                   void **pool_ptr, void **meta_ptr);
int ps_route_peers(ps_ctx *ctx, int nparts, void *const *pool_ptrs, void *const *meta_ptrs);
/* One process, several contexts (one per rank, any devices): register the receive pools of ranks[0..nparts-1]
 * (ranks[d] has done ps_route_setup(nparts, d, ...); ranks[my_rank] == ctx) and enable peer access from ctx's
 * device to every other device among them. Call after every rank's ps_route_setup, before ps_route_begin.
 * PS_ERR_STATE: a rank set up with another nparts or rank index, or without a pool; PS_ERR_ARG: more than
 * PART_MAX ranks, or two devices without peer access. */
int ps_route_connect(ps_ctx *ctx, int nparts, ps_ctx *const *ranks);
int ps_route_begin(ps_ctx *ctx);
int ps_route_scatter(ps_ctx *ctx);
int ps_route_build(ps_ctx *ctx, uint64_t *n_union, int *overflow);
/* CUDA IPC plumbing for one process per GPU: 64-byte handle of a device allocation of this context,
 * mapping of a peer's handle (cached per handle), and release of all mappings. */
int ps_ipc_export(ps_ctx *ctx, const void *dev_ptr, uint8_t handle[64]);
int ps_ipc_open(ps_ctx *ctx, const uint8_t handle[64], void **ptr);
int ps_ipc_close_all(ps_ctx *ctx);
/*
 * nq-quantiles (nq - 1 values) of one sample's sorted distinct k-mers: balanced boundaries for
 * ps_set_range when the k-mer space is cut into nq ranges (GPUs or memory partitions).
 */
int ps_sample_quantiles(ps_ctx *ctx, int idx, int nq, uint64_t *out);

/*
 * -w sample weights (Mash distances + neighbour joining + GSC, modeling.py:386-503) on the device.
 *
 * Part 1: MinHash sketches of samples first_idx..first_idx+count-1 from their decoded streams (samples must be
 * present; any job k / cutoff; FASTQ and cutoff > 1 samples keep their streams too): the s smallest distinct h1 of
 * MurmurHash3_x64_128(seed) over the upper-case text of every canonical k-mer, as `mash sketch -r -k k -s s -S seed`.
 * hashes[i*s + j] ascending, n_hashes[i] <= s (entries past n_hashes[i] are 0). k 1..32, s 1..4096.
 * Replaces: Samples.get_mash_sketches -> `mash sketch -r` (modeling.py:386-390).
 */
int ps_mash_sketch(ps_ctx *ctx, int first_idx, int count, int k, int s, uint32_t seed,
                   uint64_t *hashes, uint32_t *n_hashes);
/*
 * Part 2: shared_denom[i*n + j] = shared << 16 | denom for all ordered pairs of n sketches laid out as
 * ps_mash_sketch returns them (host or device input): denom = min(s, |A u B|), shared = elements of A n B among the
 * denom smallest of A u B. Replaces: `mash paste` + `mash dist` (modeling.py:404-412).
 */
int ps_mash_pairs(ps_ctx *ctx, int n, int s, const uint64_t *hashes, const uint32_t *n_hashes,
                  uint32_t *shared_denom);
/*
 * Part 3: neighbour joining (Biopython 1.76 as restated in weights.py) on a symmetric n x n FP64 matrix (host or
 * device), n 3..65535. join[2t], join[2t+1] = list positions (mi, mj) joined at step t < n-2; branch[2t],
 * branch[2t+1] = their branch lengths; branch[2(n-2)] = the last remaining distance.
 * Replaces: DistanceTreeConstructor.nj (modeling.py:446-452).
 * None of the three touches the job's union, matrix, survivors or k-mer range.
 */
int ps_neighbor_joining(ps_ctx *ctx, int n, const double *dm, int32_t *join, double *branch);

/* Instrumentation: the CUDA stream all work runs on; kernel launch counter; per-kernel
 * CUDA-event timing (enable, run, then read name / launches / total ms per kernel). */
void *ps_stream(ps_ctx *ctx);
uint64_t ps_launch_count(ps_ctx *ctx);
int ps_profile_enable(ps_ctx *ctx, int on);
int ps_profile_count(ps_ctx *ctx);
int ps_profile_get(ps_ctx *ctx, int i, const char **name, uint64_t *launches,
                   double *total_ms, double *alg_bytes);
int ps_profile_reset(ps_ctx *ctx);
/* Device memory currently held by the context, bytes. */
uint64_t ps_device_bytes(ps_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* PSKMER_H */
