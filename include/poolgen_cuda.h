/*
 * poolgen_cuda.h -- C ABI of the B200 (sm_100a) per-locus GWAS scan library (libpoolgen_cuda.so).
 *
 * This is the drop-in boundary for ONE hot path of jeffersonfparil/poolgen: the per-locus
 * callbacks that `ChunkyReadAnalyseWrite::read_analyse_write` invokes for every line of a sync
 * file (reference: src/base/structs_and_traits.rs:245-265, impls src/base/sync.rs:606-786 and
 * 788-970), i.e.
 *      gwas::ols_iterate          src/gwas/ols.rs:201-276            PG_KIND_OLS
 *      gwas::correlation          src/gwas/correlation_test.rs:73-129 PG_KIND_CORR
 *      tables::chisq              src/tables/chisq_test.rs:5-47       PG_KIND_CHISQ
 *      tables::fisher             src/tables/fisher_exact_test.rs:32-130 PG_KIND_FISHER
 * and the whole-matrix entry `ols_with_covariate` (src/gwas/ols.rs:278-436) through the pg_kin_*
 * functions.  The per-locus callback `Fn(&mut T, &FilterStats) -> Option<String>` becomes a
 * per-BATCH call: the reader threads parse their byte range (src/base/sync.rs:827-868) into a slab
 * of counts, hand the slab over, and format the returned numeric records with the reference's own
 * rounding rules (src/base/helpers.rs:103-117).  INTEGRATION.md shows the Rust `extern "C"` stub.
 *
 * Conventions
 *   - plain C, no C++ types, no exceptions cross this boundary; every function returns an int
 *     (PG_OK = 0, negative = error class); the message is available from pg_last_error().
 *   - one pg_ctx per GPU (one process or one thread per GPU); all functions taking the same
 *     pg_batch must be called from one thread at a time; different batches are independent.
 *   - allele codes follow the sync column order A:T:C:G:N:D = 0..5 (src/base/sync.rs:134-137).
 *   - per-locus failures are DATA (status codes), never errors.
 *   - there is no CPU fallback: every entry point fails with PG_ERR_CUDA when no sm_100 device
 *     is usable.
 */
#ifndef POOLGEN_CUDA_H
#define POOLGEN_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_ABI_VERSION 1

enum { PG_OK = 0, PG_ERR_ARG = -1, PG_ERR_CUDA = -2, PG_ERR_STATE = -3, PG_ERR_UNSUPPORTED = -4, PG_ERR_NCCL = -5 };

/* the per-locus analyses (callbacks); 4 is PG_KIND_OLS_KINSHIP, a header selector of the writer.
 * PG_KIND_MLE: gwas::mle_iterate (src/gwas/mle.rs:232-305), phenotypes as for PG_KIND_OLS; records: statistic = beta,
 *   stats[1] = v_b (a variance, mle.rs:150-154), t = beta / v_b (sic, mle.rs:176), p.
 * PG_KIND_GWALPHA_LS / _ML: gwas::gwalpha_ls / gwalpha_ml (src/gwas/gwalpha.rs:282-386); `phen` of pg_scan_open is the
 *   gwalpha_fmt matrix (rows x 3 row-major: column 0 bins, column 1 q, column 2 = sig, MIN, MAX then -inf,
 *   src/base/phen.rs) and `k` its number of rows; records: n_phen = 1, statistic = alpha, stats[1] = p_a.
 * Both minimise with argmin's Nelder-Mead capped at 1,000 iterations: results agree with the reference to the
 * solver's convergence, not to 1e-9 (DESIGN.md 11). */
enum { PG_KIND_OLS = 0, PG_KIND_CORR = 1, PG_KIND_CHISQ = 2, PG_KIND_FISHER = 3, PG_KIND_MLE = 5, PG_KIND_GWALPHA_LS = 6,
       PG_KIND_GWALPHA_ML = 7 };

/* per-locus status, = what the reference callback returned */
enum {
    PG_LOCUS_FILTERED = 0,    /* None: LocusCounts::filter dropped the locus (src/base/sync.rs:195-303) */
    PG_LOCUS_OK = 1,          /* Some(line) */
    PG_LOCUS_FAILED = 2,      /* None: the regression could not be solved (src/gwas/ols.rs:250-253) */
    PG_LOCUS_UNSUPPORTED = 3, /* shape the device path does not implement (mle_iter with fewer pools than coefficients) */
    PG_LOCUS_PANIC = 4        /* the reference would panic on this locus (assert / unwrap) */
};

#define PG_MAX_ALLELES 6
#define PG_MAX_SLOTS 5 /* output rows per locus = kept alleles - 1 <= 5 */

typedef struct pg_ctx pg_ctx;
typedef struct pg_scan pg_scan;
typedef struct pg_batch pg_batch;

/* FilterStats (src/base/structs_and_traits.rs:69-78); only the fields the sync path reads.
 * pool_sizes are taken as handed over by the phenotype loader, i.e. already normalised to sum 1
 * (src/base/phen.rs:82-84); the library re-derives s_i / sum(s) exactly as src/base/sync.rs:262-270. */
typedef struct {
    int32_t remove_ns;             /* !--keep-ns */
    uint64_t min_coverage_depth;   /* --min-coverage-depth */
    double min_allele_frequency;   /* --min-allele-frequency */
    double max_missingness_rate;   /* --max-missingness-rate */
    int32_t n_pool_sizes;
    const double *pool_sizes;
} pg_filter;

/* Numeric records of one batch, host pointers owned by the library (pinned), valid until the next
 * download/destroy of that batch.  L = n_loci, S = n_slots (= n_alleles_dev - 1), k = n_phen.
 *   meta[l]      byte0 status, byte1 n_out (rows for this locus), byte 2+s allele code of row s
 *   freq_mean[l*S+s]            mean frequency of that allele            (ols.rs:265-268 / correlation_test.rs:119)
 *   stats[((l*S+s)*k+j)*4 + c]  c=0 statistic (beta | r rounded to 7 digits, correlation_test.rs:70)
 *                               c=1 standard error of beta | unrounded r
 *                               c=2 t
 *                               c=3 p-value
 * CHISQ / FISHER: S = 1, k = 1, n_out = number of kept alleles, allele codes of ALL kept alleles in
 * bytes 2.., stats[l*4+0] = chi2 | p_observed, stats[l*4+3] = p-value, freq_mean unused. */
typedef struct {
    int64_t n_loci;
    int32_t n_slots;
    int32_t n_phen;
    const uint64_t *meta;
    const double *freq_mean;
    const double *stats;
} pg_results;

/* ---- context ------------------------------------------------------------------------------- */
int pg_abi_version(void);
int pg_init(int device, pg_ctx **out);
void pg_destroy(pg_ctx *ctx);
const char *pg_last_error(const pg_ctx *ctx); /* ctx may be NULL: last error of a failed pg_init */
int pg_device_info(pg_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);
/* free and total device memory at the time of the call (cudaMemGetInfo): the GPU may be shared, so a budget for device
 * blocks is taken from free_bytes, not from the card's total */
int pg_device_mem_info(pg_ctx *ctx, size_t *free_bytes, size_t *total_bytes);
/* pinned host slabs the reader threads parse into */
int pg_pinned_alloc(pg_ctx *ctx, size_t bytes, void **out);
int pg_pinned_free(pg_ctx *ctx, void *p);

/* ---- scan configuration = (callback, FilterStats, phenotypes) --------------------------------
 * n_alleles / allele_codes name the count columns the caller ships per pool (a subset of the six
 * sync columns, in sync order).  When filter->remove_ns is set a column coded N(4) is dropped on
 * the device exactly like src/base/sync.rs:200-213.
 * phen: n_pools x k row-major f64 (Phen.phen_matrix, src/base/phen.rs:86-97); NULL/0 for the table tests. */
int pg_scan_open(pg_ctx *ctx, int kind, const pg_filter *filter, int n_pools, int n_alleles,
                 const uint8_t *allele_codes, const double *phen, int k, pg_scan **out);
int pg_scan_close(pg_scan *scan);

/* ---- batches: a device-resident block of loci + its results ---------------------------------- */
int pg_batch_create(pg_scan *scan, int64_t capacity_loci, pg_batch **out);
int pg_batch_destroy(pg_batch *b);
/* host -> device, asynchronous on the batch's stream.
 * counts: u32 [locus][allele][pool] (pool fastest), the parsed LocusCounts.matrix transposed. */
int pg_batch_upload_counts(pg_batch *b, const uint32_t *counts, int64_t n_loci);
/* same, 16-bit counts (every count < 65536): half the PCIe bytes */
int pg_batch_upload_counts_u16(pg_batch *b, const uint16_t *counts, int64_t n_loci);
/* same, 8-bit counts (every count < 256, typical for pool-seq depths below 255): a quarter of the PCIe bytes */
int pg_batch_upload_counts_u8(pg_batch *b, const uint8_t *counts, int64_t n_loci);
/* f64 first-stage frequency matrix, column-major n_pools x n_alleles per locus ([locus][allele][pool],
 * N column already removed, NaN where the pool has no coverage) + per-pool depth [locus][pool].
 * OLS / CORR only. */
int pg_batch_upload_freq(pg_batch *b, const double *freq, const uint32_t *depth, int64_t n_loci);
/* sync TEXT on the fast path: a line-aligned chunk of a sync file (chr \t pos \t ref \t A:T:C:G:N:D per pool, as the
 * chunk readers hand lines to `lparse`, src/base/sync.rs:100-156, 827-868) is copied to the device as it is and parsed
 * there.  Commented lines and lines whose position is not an integer are skipped like the reference skips them; a pool
 * count that differs from the scan's, or a malformed pool field (the reference panics), is PG_ERR_ARG with the byte
 * offset in the message.  The scan must have been opened with the six sync columns (codes 0..5).  Synchronises the
 * batch's stream.  pg_batch_text_labels: per parsed locus the byte offset of its line in the chunk (chromosome and
 * position text for the writer) and the parsed position, host pointers valid until the next text upload. */
int pg_batch_upload_sync_text(pg_batch *b, const char *text, size_t n_bytes, int64_t *n_loci);
int pg_batch_text_labels(pg_batch *b, const uint64_t **line_offsets, const uint64_t **positions);
/* synthetic counts generated on the device (integer hash; pg_synth_counts_host replays it bit for bit) */
int pg_batch_synth(pg_batch *b, uint64_t seed, int64_t first_locus, int64_t n_loci);
/* launch the scan kernel over the loci resident in the batch (asynchronous) */
int pg_batch_run(pg_batch *b);
/* device -> pinned host copy of the result records (asynchronous), then pg_batch_sync + pg_batch_results */
int pg_batch_download(pg_batch *b);
int pg_batch_sync(pg_batch *b);
int pg_batch_results(pg_batch *b, pg_results *out);
/* timing helper: `iters` back-to-back pg_batch_run launches bracketed by CUDA events on the batch's
 * stream; returns the total milliseconds and how many kernels were launched */
int pg_batch_time_runs(pg_batch *b, int iters, float *ms_total, int *n_launches);
/* device bytes one launch reads as input and writes as results (for traffic accounting) */
int pg_batch_bytes(pg_batch *b, size_t *input_bytes, size_t *result_bytes);

/* ---- streaming convenience used by the reader threads (src/base/sync.rs:917-939): submit a slab,
 * get a ticket, collect the records later; up to PG_STREAM_DEPTH slabs are in flight so the H2D
 * copy of slab i+1 overlaps the scan of slab i and the D2H copy of slab i-1. ---------------------- */
#define PG_STREAM_DEPTH 3
int pg_scan_stream_begin(pg_scan *scan, int64_t max_loci_per_slab);
int pg_scan_submit_counts(pg_scan *scan, const uint32_t *counts, int64_t n_loci, int *ticket);
int pg_scan_submit_counts_u16(pg_scan *scan, const uint16_t *counts, int64_t n_loci, int *ticket);
int pg_scan_submit_counts_u8(pg_scan *scan, const uint8_t *counts, int64_t n_loci, int *ticket);
int pg_scan_submit_freq(pg_scan *scan, const double *freq, const uint32_t *depth, int64_t n_loci, int *ticket);
/* text slabs: the copy and the device-side parse are enqueued and the call returns; the scan of a slab is launched by
 * the NEXT submit (or by its collect), once the parse has told the host how many loci the chunk holds -- so the copy of
 * slab i+1 overlaps the parse of slab i.  `text` must stay valid and unchanged until the ticket has been collected.
 * n_loci may be NULL; when it is not, the call waits for this slab's parse (no deferral).  Errors of a deferred slab
 * (pool count, malformed field) surface from the call that finishes it. */
int pg_scan_submit_sync_text(pg_scan *scan, const char *text, size_t n_bytes, int *ticket, int64_t *n_loci);
int pg_scan_collect(pg_scan *scan, int ticket, pg_results *out);
/* labels of a slab submitted as text (see pg_batch_text_labels), valid until the ticket's slab is submitted again */
int pg_scan_text_labels(pg_scan *scan, int ticket, const uint64_t **line_offsets, const uint64_t **positions);

/* ---- ols_iter_with_kinship: ols_with_covariate (src/gwas/ols.rs:278-436) over a device-resident block of allele
 * columns of GenotypesAndPhenotypes.intercept_and_allele_frequencies[:, 1..] (src/base/sync.rs:1106-1179).
 * One pg_kin per GPU holds that GPU's column shard.  Sequence: append columns -> pg_kin_gram (partial G G') ->
 * [sum the partials over the GPUs: pg_kin_allreduce, below] ->
 * pg_kin_eig_select (K = sum / P_total, eigen-decomposition, number of PCs by the reference's rule) ->
 * pg_kin_covar_scan (beta, var(beta), p of the allele coefficient with X = [1 | PCs | g], one record per column
 * and phenotype; the caller writes them phenotype-outer / column-inner like src/gwas/ols.rs:410-433). ----------- */
typedef struct pg_kin pg_kin;
int pg_kin_open(pg_ctx *ctx, int n_pools, int64_t max_columns, pg_kin **out);
int pg_kin_close(pg_kin *kin);
int pg_kin_reset(pg_kin *kin);
int64_t pg_kin_columns(pg_kin *kin);
/* host f64 allele columns, column-major [P_add][n_pools] */
int pg_kin_append_columns(pg_kin *kin, const double *cols, int64_t P_add);
/* a slab of parsed loci (u32 [locus][allele][pool]) through LoadAll::load semantics (src/base/sync.rs:973-1104): filter,
 * renormalised frequencies of the kept alleles, with keep_p_minus_1 the sort by column sum and the drop of the major
 * allele; every kept allele becomes one column.  pg_kin_last_labels returns (locus ordinal in the slab, allele code)
 * of the columns the last call appended. */
int pg_kin_append_counts(pg_kin *kin, const pg_filter *filter, int n_alleles, const uint8_t *allele_codes,
                         const uint32_t *counts, int64_t n_loci, int keep_p_minus_1, int64_t *n_cols_added);
int pg_kin_last_labels(pg_kin *kin, int64_t n_cols, int64_t *col_locus, uint8_t *col_allele);
/* the same from a line-aligned chunk of sync TEXT (see pg_batch_upload_sync_text), parsed on the device straight into
 * the loader's count slab; max_loci bounds the loci of a chunk.  pg_kin_text_labels: byte offset of each parsed locus'
 * line and its position (host pointers valid until the next text append) -- col_locus of pg_kin_last_labels indexes them. */
int pg_kin_append_sync_text(pg_kin *kin, const pg_filter *filter, const char *text, size_t n_bytes, int64_t max_loci,
                            int keep_p_minus_1, int64_t *n_loci, int64_t *n_cols_added);
int pg_kin_text_labels(pg_kin *kin, const uint64_t **line_offsets, const uint64_t **positions);
/* sync2csv rows formatted on the device from the columns the LAST pg_kin_append_sync_text added (column 0 = its first
 * column): columns [first, first + count), one row each, equal byte for byte to pg_format_frequency_rows over the same
 * columns, their pg_kin_last_labels and the text labels of that append with locus_order = NULL
 * (`chr,pos,allele,f_1,...,f_n\n`, every f through parse_f64_roundup_and_own(x, 6)).  The rows are copied to `out`
 * (pinned host memory for a full-rate copy); the call stops at the last whole row that fits `capacity` and returns the
 * rows done and their bytes, so a caller continues at first + *n_rows.  A capacity below one row is PG_ERR_ARG.
 * PG_ERR_STATE when the last append (or a reset) was not from text; PG_ERR_UNSUPPORTED, nothing written, when a value
 * of the range is infinite or has |x * 1e6| >= 9e14 (the loader's frequencies never do; pg_format_frequency_rows prints
 * them).  Synchronises the handle's stream. */
int pg_kin_format_frequency_rows(pg_kin *kin, int64_t first, int64_t count, char *out, size_t capacity, size_t *n_bytes,
                                 int64_t *n_rows);
/* synthetic biallelic columns (two per locus) generated on the device from the integer-hash workload */
int pg_kin_synth(pg_kin *kin, uint64_t seed, int64_t first_locus, int64_t n_loci);
int pg_kin_get_columns(pg_kin *kin, int64_t first, int64_t count, double *out /* [count][n_pools] */);
/* partial Gram matrix of the resident columns (FP64 tensor cores), asynchronous: K = G G' */
int pg_kin_gram(pg_kin *kin);
/* K += G G' of the resident columns, asynchronous like pg_kin_gram.  Columns beyond one device's memory are taken in
 * blocks: pg_kin_gram on block 1, then pg_kin_reset + load + pg_kin_gram_accumulate for blocks 2..B (pg_kin_reset
 * keeps K), then pg_kin_eig_select with P_total = the columns of all blocks.  Each slice sum is added to K in a fixed
 * order and both triangles get the same value: K is exactly symmetric and a given split is bit-repeatable.  Composes
 * with pg_kin_allreduce: each GPU accumulates its own blocks, the all-reduce sums the GPUs' totals. */
int pg_kin_gram_accumulate(pg_kin *kin);
int pg_kin_gram_time(pg_kin *kin, int iters, float *ms_total);
int pg_kin_partial(pg_kin *kin, double **device_ptr, size_t *n_elems); /* n_pools x n_pools, synchronises */
int pg_kin_partial_get(pg_kin *kin, double *out_host);
int pg_kin_partial_set(pg_kin *kin, const double *in_host);
/* P_total = 0: the column count pg_kin_allreduce summed (or, without an all-reduce, the resident columns) */
int pg_kin_eig_select(pg_kin *kin, int64_t P_total, double variance_explained, int *n_eigenvecs);
int pg_kin_eigvals(pg_kin *kin, double *out, int count); /* K's eigenvalues, high to low */
int pg_kin_set_covariates(pg_kin *kin, const double *cov /* n_pools x m row-major */, int m);
/* phen n_pools x k row-major; results host pointers (library-owned, pinned), each [k][columns];
 * iters > 0 additionally times `iters` back-to-back launches with CUDA events */
int pg_kin_covar_scan(pg_kin *kin, const double *phen, int k, int iters, float *ms_total, const double **beta,
                      const double **var, const double **pval);
/* mle_iter_with_kinship: mle_with_covariate (src/gwas/mle.rs:307-463; call site src/main.rs:316-326) over the same
 * resident columns and covariates -- per (column, phenotype) the maximum-likelihood fit of y on [1 | PCs | g] by the
 * reference's Nelder-Mead search (mle.rs:85-114), v_b = sigma2 [(X'X)^-1]_gg, t = beta / v_b (sic, mle.rs:176),
 * p from Student-t(n - 1); NaN where X'X has no inverse.  Same result layout as pg_kin_covar_scan, same rows
 * (pg_format_kinship_rows).  At most 13 covariates (a simplex of 16 parameters) and 16 phenotypes per call;
 * PG_ERR_UNSUPPORTED for the n < 2 + m form.  ms: kernel time of the scan. */
int pg_kin_mle_scan(pg_kin *kin, const double *phen, int k, float *ms, const double **beta, const double **var,
                    const double **pval);

/* ---- several GPUs behind the ABI (SURVEY.md 8b / 8e) -----------------------------------------------------------------
 * The reference runs every analysis in one process (src/main.rs:246-298).  The per-locus scans shard over loci with no
 * exchange step: pg_shard_range names the contiguous range of a rank (earlier ranks take the larger shards; rank order
 * = file order, like the reader threads' contiguous byte ranges, src/base/helpers.rs:74-91).  ols_with_covariate has
 * ONE exchange step: `g.dot(&g.t())` (src/gwas/ols.rs:295) over column shards is the sum of the per-GPU partial Gram
 * matrices -- pg_kin_allreduce (NCCL all-reduce over NVLink on the handles' own device buffers and streams; the column
 * counts are summed in the same group).  The communicator is created by the library:
 *   pg_init_multi        one process drives n GPUs (what the Rust CLI does): n contexts + ncclCommInitAll
 *   pg_comm_unique_id /  one process per GPU: rank 0 obtains the id, the host ships the PG_COMM_ID_BYTES bytes to the
 *   pg_comm_init_rank    other ranks however it likes (a file, MPI, torch.distributed), every rank joins
 * kins[i] belongs to local rank i of the communicator.  After the all-reduce every handle holds the total;
 * pg_kin_eig_select(kin, 0, ...) then uses the summed column count.  pg_kin_copy_covariates hands the outcome of one
 * eigen step to the other handles of a process (the step is replicated work).  NCCL is loaded on first use. */
typedef struct pg_comm pg_comm;
#define PG_COMM_ID_BYTES 128
int pg_shard_range(int64_t total, int rank, int world, int64_t *begin, int64_t *end);
int pg_nccl_version(int *version);
int pg_init_multi(const int *devices, int n, pg_ctx **ctxs_out /* [n] */, pg_comm **comm_out);
int pg_comm_unique_id(uint8_t *id /* [PG_COMM_ID_BYTES] */);
int pg_comm_init_rank(pg_ctx *ctx, const uint8_t *id, int rank, int world, pg_comm **out);
int pg_comm_info(const pg_comm *comm, int *world, int *n_local, int *first_rank);
int pg_comm_destroy(pg_comm *comm); /* the contexts of pg_init_multi are destroyed by the caller (pg_destroy) */
/* ms (optional): device time of the exchange step, CUDA events on kins[0]'s stream */
int pg_kin_allreduce(pg_comm *comm, pg_kin *const *kins, int n_local, int64_t *P_total, float *ms);
int pg_kin_copy_covariates(pg_kin *dst, const pg_kin *src);

/* ---- the reference's CSV rows from the numeric records (SURVEY.md 8f-2; host code, threads over locus ranges) -------
 * Replaces the string building of the per-locus callbacks (src/gwas/ols.rs:255-275, src/gwas/correlation_test.rs:113-128,
 * src/tables/chisq_test.rs:36-46, src/tables/fisher_exact_test.rs:118-129) and of ols_with_covariate
 * (src/gwas/ols.rs:409-433): numbers as Rust's f64::to_string() prints them, rounded with
 * parse_f64_roundup_and_own (src/base/helpers.rs:103-117) where the reference rounds.  Only loci with status
 * PG_LOCUS_OK produce rows, in locus order (= file order within the chunk, src/base/sync.rs:953-967). */
#define PG_KIND_OLS_KINSHIP 4 /* header selector only */
typedef struct {
    const uint64_t *positions;    /* [n_loci] */
    const char *text;             /* the sync text chunk the loci were parsed from, or NULL */
    const uint64_t *line_offsets; /* with text: [n_loci] byte offset of the locus' line (pg_batch_text_labels);
                                     the chromosome is the text up to the first tab */
    const char *const *chr_names; /* without text: table of NUL-terminated chromosome names ... */
    const uint32_t *chr_index;    /* ... and [n_loci] indices into it */
} pg_row_labels;
/* the header line of the output file (src/base/sync.rs:766,950, src/gwas/ols.rs:409) */
int pg_format_header(int kind, char *out, size_t capacity, size_t *n_bytes);
/* rows of `res` (OLS / CORR / CHISQ / FISHER); *n_bytes = bytes written, or needed when capacity is too small
 * (PG_ERR_ARG, nothing written) */
int pg_format_rows(int kind, const pg_results *res, const pg_row_labels *labels, int n_threads, char *out,
                   size_t capacity, size_t *n_bytes);
/* the same with options.  PG_FORMAT_EXACT_P (OLS / CORR): the printed p-value is re-derived on the host from the record's
 * t statistic with the reference's own arithmetic -- statrs' StudentsT::cdf through its Lentz continued fraction, df =
 * n_pools - 1 (src/gwas/ols.rs:139,153) or n_pools - 2 (src/gwas/correlation_test.rs:65-66) -- instead of the device's
 * table value (accurate to ~1e-12, inside the record tolerance of 1e-6 but enough to move a 12th printed decimal).  Rows
 * then differ from the reference's only where the t statistic itself differs in its last digits.  About 0.3 us per row. */
#define PG_FORMAT_EXACT_P 1
int pg_format_rows_ex(int kind, const pg_results *res, const pg_row_labels *labels, int flags, int n_pools,
                      int n_threads, char *out, size_t capacity, size_t *n_bytes);
/* rows of ols_iter_with_kinship: phenotype outer, column inner; beta / pval as pg_kin_covar_scan returns them
 * ([k][n_columns]); chromosome / position / allele are indexed by the column ordinal exactly like
 * src/gwas/ols.rs:421-424 indexes the label vectors of GenotypesAndPhenotypes (whose entry 0 is "intercept") */
int pg_format_kinship_rows(int64_t n_columns, int k, const char *const *chromosome, const uint64_t *position,
                           const char *const *allele, const double *beta, const double *pval, int n_threads,
                           char *out, size_t capacity, size_t *n_bytes);
/* sync2csv (SaveCsv::write_csv, src/base/sync.rs:1182-1262) on top of the column loader (pg_kin_append_counts +
 * pg_kin_get_columns + pg_kin_last_labels): one row per allele column, `chr,pos,allele,f_1,...,f_n` with every
 * frequency through parse_f64_roundup_and_own(x, 6).  labels are indexed by the locus ordinal col_locus[c]; columns must
 * be grouped by ascending locus ordinal (as the loader emits them).  locus_order (optional) lists the locus ordinals in
 * output order -- pg_sort_loci gives the reference's order, a stable sort by (chromosome bytes, position)
 * (src/base/sync.rs:1092-1101). */
int pg_sort_loci(const pg_row_labels *labels, int64_t n_loci, int64_t *order_out);
int pg_format_frequency_header(const char *const *pool_names, int n_pools, char *out, size_t capacity, size_t *n_bytes);
int pg_format_frequency_rows(int64_t n_columns, int n_pools, const double *columns /* [n_columns][n_pools] */,
                             const int64_t *col_locus, const uint8_t *col_allele, const pg_row_labels *labels,
                             const int64_t *locus_order, int64_t n_order, int n_threads, char *out, size_t capacity,
                             size_t *n_bytes);
/* one number: n_digits > 0 = parse_f64_roundup_and_own(x, n_digits), 0 = f64::to_string(); returns the length */
int pg_format_f64(double x, int n_digits, char *out, size_t capacity);

#ifdef __cplusplus
}
#endif
#endif
