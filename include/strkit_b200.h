/*
 * strkit_b200.h -- C ABI of the B200-native replacement for STRkit's per-read repeat-count
 * hot path.  Plain C: pointers, sizes, int status codes (0 = OK); no exceptions cross the
 * boundary; strk_last_error() returns a thread-local message for the last non-zero status.
 *
 * What each entry point replaces in the reference (paths relative to the reference checkout):
 *
 *   strk_count_reads / strk_batch_*   the per-read loop of call_locus (strkit/call/call_locus.py:
 *                                     1079,1129-1161) around strkit.call.repeats.get_repeat_count
 *                                     (strkit/call/repeats.py:47-70), i.e. the PyO3 binding
 *                                     strkit_rust_ext.get_repeat_count(start_count, tr_seq, fl, fr,
 *                                     motif, max_iters, local_search_range, step_size,
 *                                     use_shortcuts=False) (repeats.py:58-68), batched over the
 *                                     reads of many loci (replacing the worker pool's per-locus
 *                                     calls, strkit/call/call_sample.py:103-157).
 *   strk_score_tables                 the candidate scoring inside that search: the alignment of
 *                                     fl + motif*n + fr against the profile of fl + tr + fr for a
 *                                     whole window of n at once (parasail sg*_scan_profile_sat).
 *   strk_ref_boundary_tables          score_ref_boundaries (repeats.py:23-43): the two
 *                                     parasail.sg_qe_scan_profile_sat calls, for a window of n.
 *   strk_ref_counts                   get_ref_repeat_count (repeats.py:73-192), batched over loci.
 *   strk_init(matrix, gap...)         strkit/call/align_matrix.py:15-44 (dna_matrix, indel_penalty)
 *                                     and parasail.profile_create_sat (repeats.py:92-93).
 *
 * Sequences are passed as they are in the reference: ASCII bytes (any case; IUPAC codes, the
 * low-quality wildcard 'X', unknown bytes -> parasail's wildcard column).  The device encodes.
 *
 * Ownership: every buffer is caller-allocated and caller-freed; the library keeps no host
 * pointer after a call returns.  Threading: one context per GPU per host thread; calls on one
 * context are not re-entrant.  There is no CPU fallback: without a CUDA device strk_init fails.
 */
#ifndef STRKIT_B200_H
#define STRKIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct strk_ctx strk_ctx;
typedef struct strk_batch strk_batch;

/* status codes */
#define STRK_OK 0
#define STRK_ERR_ARG 1     /* invalid argument (null pointer, negative size, empty sequence, ...)  */
#define STRK_ERR_CUDA 2    /* CUDA runtime error (message has the detail)                          */
#define STRK_ERR_NOMEM 3   /* host or device allocation failed                                     */
#define STRK_ERR_UNSUPPORTED 4 /* e.g. gap_open != gap_extend (the reference always passes 5, 5)   */
#define STRK_ERR_SEARCH 5  /* the search scored nothing (reference raises ValueError)              */

/* free-end flags of the semi-global alignment; s1 = db (the profiled sequence), s2 = candidate */
#define STRK_S1_BEG_FREE 1
#define STRK_S1_END_FREE 2
#define STRK_S2_BEG_FREE 4
#define STRK_S2_END_FREE 8
#define STRK_MODE_SG 15   /* parasail "sg"    */
#define STRK_MODE_SG_QE 2 /* parasail "sg_qe" */

/* tie-break switches of the read-path search (0 = the in-tree Python semantics) */
#define STRK_TIE_WINDOW_LAST 1
#define STRK_TIE_FINAL_LAST 2
/* search-policy switches of the same flag word: hypotheses about the Rust body of strkit_rust_ext.get_repeat_count,
 * which is not in the reference tree (strkit/call/repeat_count_params.py:13: the initial local search range "can be
 * narrowed within the get_repeat_count fn").  0 = range fixed, as in the in-tree search of repeats.py:100-151. */
#define STRK_SEARCH_NARROW_FIRST 4 /* range becomes 1 after the first (direction 0) window */
#define STRK_SEARCH_NARROW_HALVE 8 /* range is halved (not below 1) after every window     */

#define STRK_NSYM 17

/* kernel selection for strk_batch_run / strk_count_reads and the raw tables (strk_score_tables,
 * strk_ref_boundary_tables) */
#define STRK_KERNEL_AUTO 0    /* packed u16x2 kernel where its preconditions hold, else general */
#define STRK_KERNEL_GENERAL 1 /* int32 general kernel for everything (any length / alphabet)    */

const char *strk_last_error(void);
const char *strk_version(void);

/* Number of visible CUDA devices (0 when there is none; never fails). */
int strk_device_count(void);

/* Create a context on `device`.  matrix = 17x17 row-major substitution scores (align_matrix.py),
 * end_flags = free ends of the read-path alignment (STRK_MODE_SG by default in the wrappers),
 * tie_flags = STRK_TIE_* switches. */
int strk_init(int device, const int8_t matrix[STRK_NSYM * STRK_NSYM], int gap_open, int gap_extend, int end_flags,
              int tie_flags, strk_ctx **ctx);
int strk_destroy(strk_ctx *ctx);
/* Wait for everything queued on the context's streams (SURVEY 8b minimum set).  Every entry point of this header
 * returns with its results in the caller's buffers, so this only matters after strk_batch_run on a caller stream. */
int strk_sync(strk_ctx *ctx);

/* Pin / unpin a caller-owned host buffer so that copies are asynchronous DMA. */
int strk_host_register(void *ptr, uint64_t bytes);
int strk_host_unregister(void *ptr);

/*
 * A batch = the reads of n_loci loci, in locus order and read order (the order matters: the start
 * guess of read k uses the results of reads < k of the same locus, call_locus.py:1129-1161).
 *   arena        ASCII bytes holding every sequence
 *   seq_off[r]   offset of read r's concatenation fl + tr + fr (contiguous)
 *   lens[3r..]   {len(fl), len(tr), len(fr)}
 *   est_cn[r]    get_est_copy_num() of the read (call_locus.py:1129)
 *   read_begin   n_loci + 1 prefix offsets into the read arrays
 *   motif_off/motif_len  per locus, into the same arena
 * strk_batch_upload copies everything to the device (H2D) and builds the work plan.
 */
int strk_batch_upload(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                      const int32_t *lens, const int32_t *est_cn, int64_t n_reads, const int64_t *read_begin,
                      const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci, strk_batch **batch);

/* An empty, reusable batch and its (re)fill: strk_batch_fill replaces the contents and recycles the device
 * buffers (no cudaMalloc once they have grown to the block size).  strk_batch_upload = create + fill.
 * A host thread that keeps two contexts on one GPU can overlap the H2D copy of locus block i+1 (fill on
 * context B) with the kernels of block i (run on context A): the reference's worker pool streams locus
 * blocks the same way (strkit/call/call_sample.py:413-420). */
int strk_batch_create(strk_ctx *ctx, strk_batch **batch);
int strk_batch_fill(strk_ctx *ctx, strk_batch *batch, const uint8_t *arena, uint64_t arena_bytes,
                    const uint64_t *seq_off, const int32_t *lens, const int32_t *est_cn, int64_t n_reads,
                    const int64_t *read_begin, const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci);

/* Arena formats.  STRK_ARENA_ASCII: one byte per symbol, as the reference passes its strings.  STRK_ARENA_NIBBLE: two
 * symbols per byte (low nibble first), code = index into the reference's alphabet "ACGTRYSWKMBDHVNX"
 * (align_matrix.py:25-26): half the host-to-device bytes of a block.  arena_bytes counts packed bytes; seq_off,
 * motif_off and lens are in SYMBOLS in both formats.  Bytes outside the 16-letter alphabet (parasail's wildcard
 * column) have no nibble code: a block that holds one stays ASCII.  The device expands the packed copy (one pass of
 * 128-bit loads / stores) before any kernel stages a read. */
#define STRK_ARENA_ASCII 0
#define STRK_ARENA_NIBBLE 1
int strk_batch_fill_fmt(strk_ctx *ctx, strk_batch *batch, int arena_format, const uint8_t *arena, uint64_t arena_bytes,
                        const uint64_t *seq_off, const int32_t *lens, const int32_t *est_cn, int64_t n_reads,
                        const int64_t *read_begin, const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci);
int strk_count_reads_fmt(strk_ctx *ctx, int arena_format, const uint8_t *arena, uint64_t arena_bytes,
                         const uint64_t *seq_off, const int32_t *lens, const int32_t *est_cn, int64_t n_reads,
                         const int64_t *read_begin, const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci,
                         int max_iters, int local_search_range, int step_size, int kernel, int32_t *out);

/* Run the whole search for a resident batch: score tables (CUDA), exact replay of the reference's
 * hill-climb per locus (CUDA), widening passes for reads whose search left the table window.
 * Results stay on the device.  `stream` is a cudaStream_t (NULL = the context's own stream);
 * the call returns after the work has completed (the widening check needs the status word). */
int strk_batch_run(strk_ctx *ctx, strk_batch *batch, int max_iters, int local_search_range, int step_size,
                   int kernel, void *stream);

/* out[4r..4r+3] = {best_n, best_score, n_explored, start_count used}  (D2H). */
int strk_batch_download(strk_ctx *ctx, strk_batch *batch, int32_t *out);
int strk_batch_free(strk_ctx *ctx, strk_batch *batch);

/* Convenience: upload + run + download with host buffers (the call the Python batcher makes). */
int strk_count_reads(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                     const int32_t *lens, const int32_t *est_cn, int64_t n_reads, const int64_t *read_begin,
                     const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci, int max_iters,
                     int local_search_range, int step_size, int kernel, int32_t *out);

/* strkit_rust_ext.get_repeat_count(start_count, tr_seq, flank_left_seq, flank_right_seq, motif, max_iters,
 * local_search_range, step_size, use_shortcuts=False) (the PyO3 call at strkit/call/repeats.py:58-68), argument for
 * argument: strings with explicit lengths (no terminator needed), out4 = {best_n, best_score, n_explored,
 * best_n - start_count} = the ((n, score), n_explored, delta) the reference returns (:55-56).
 * use_shortcuts != 0 -> STRK_ERR_UNSUPPORTED (the reference always passes False). */
int strk_get_repeat_count(strk_ctx *ctx, int start_count, const char *tr_seq, int n_tr, const char *flank_left_seq,
                          int n_fl, const char *flank_right_seq, int n_fr, const char *motif, int m, int max_iters,
                          int local_search_range, int step_size, int use_shortcuts, int32_t out4[4]);

/* Raw score tables: scores[out_off[r] + (n - n_lo[r])] = alignment score of fl + motif*n + fr vs
 * fl + tr + fr for n in [n_lo[r], n_hi[r]], read r using the motif of locus motif_idx[r]. */
int strk_score_tables(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                      const int32_t *lens, const int32_t *motif_idx, const int32_t *n_lo, const int32_t *n_hi,
                      int64_t n_reads, const uint64_t *motif_off, const int32_t *motif_len, int64_t n_motifs,
                      const uint64_t *out_off, int kernel, int32_t *scores);

/* score_ref_boundaries for a window of n: out[4*(out_off[l] + n - n_lo[l]) ..] =
 * {fwd_score, fwd_end_query, rev_score, rev_end_query}  (end_query as parasail reports it;
 * r_adj = fwd_end_query + 1 - len(fl) - ref_size, repeats.py:34,41). */
int strk_ref_boundary_tables(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                             const int32_t *lens, const int32_t *n_lo, const int32_t *n_hi, int64_t n_loci,
                             const uint64_t *motif_off, const int32_t *motif_len, const uint64_t *out_off,
                             int kernel, int32_t *out);

/* get_ref_repeat_count for n_loci loci.  start_count / ref_size / rc params per locus
 * (rc_params[3l..] = {max_iters, local_search_range, step_size}, repeat_count_params.py:17-42).
 * out[8l..] = {cn, score, l_offset, r_offset, n_offset_scores, n_iters_final, new_len_fl, new_len_fr}.
 * Afterwards stats[5] (strk_get_stats) counts the loci whose search left the windows the device tried first and that
 * the host finished. */
int strk_ref_counts(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                    const int32_t *lens, const int32_t *start_count, const int32_t *ref_size,
                    const int32_t *rc_params, int64_t n_loci, const uint64_t *motif_off, const int32_t *motif_len,
                    int vcf_anchor_size, int respect_coords, int32_t *out);

/* Counters of the last strk_batch_run on this context:
 *   stats[0] executed DP cells (real cells, padding excluded)
 *   stats[1] reference-equivalent DP cells (sum over the sizes the reference search scores)
 *   stats[2] kernels launched           stats[3] DP-kernel time, ms (CUDA events on the run's stream)
 *   stats[4] replay-kernel time, ms     stats[5] widening passes run
 *   stats[6] reads handled by the packed kernel   stats[7] reads handled by the general kernel */
int strk_get_stats(strk_ctx *ctx, double stats[8]);

/*
 * call_alleles (strkit/call/allele.py:176-336), batched over loci: weighted bootstrap resampling of each locus'
 * per-read copy numbers (get_resampled_bootstrapped_reads, :126-173, separate_strands = False as both call sites
 * pass it, call_locus.py:201-214,255-268), a one- or two-component spherical Gaussian mixture per replicate
 * (fit_gmm :56-123 over sklearn.mixture.GaussianMixture: k-means++ seeding, n_init restarts, tol 1e-3, max_iter 100,
 * reg_covar 1e-6; the weight filters of :88-121; make_single_gaussian, gmm.py:72-80), then per-allele medians and
 * interpolated-inverted-CDF confidence intervals over the replicates (:295-336).
 *   cn / weights   per read, loci delimited by read_begin[n_loci + 1]; weights as the reference passes them
 *                  (normalised per locus, call_locus.py:191-192)
 *   out_i[l]       1 + 5 * n_alleles ints: modal_n, call[A], call_95_cis[A][2], call_99_cis[A][2]
 *   out_d[l]       3 * n_alleles doubles: means[A], weights[A], stdevs[A]
 *   out_status[l]  0 = bootstrapped, 1 = fewer than min_reads reads (the reference returns None),
 *                  2 = a single distinct copy number (no bootstrap, allele.py:196-214)
 *   ms_out         device time of the kernels (CUDA events), may be NULL
 * The random streams are this library's (counter-based Philox keyed by seed, locus, replicate), not numpy's:
 * results agree with the reference statistically.  n_alleles 1 and 2 are implemented here; per-locus counts up to 8
 * take the _ploidy entry below.
 * Read depth: a locus of at most 256 reads is shallow (one thread per replicate, arrays strided by the batch's
 * largest shallow locus); a locus of more reads is deep: it is resampled and fitted one warp per replicate (see
 * strk_gmm_fit_counts_deep) from ragged per-locus storage, on random streams of its own keyed by seed, locus and
 * replicate, so its rows depend neither on the chunking nor on the other loci, and shallow rows do not depend on it.
 * The rule follows from the read count alone.  A deep locus may have up to 4096 distinct copy numbers; one with more
 * is STRK_ERR_UNSUPPORTED, and the message names the locus.
 */
int strk_call_alleles(strk_ctx *ctx, const int32_t *cn, const double *weights, const int64_t *read_begin,
                      int64_t n_loci, int n_alleles, int num_bootstrap, int min_reads, int min_allele_reads,
                      int force_gm_filter, double expansion_ratio, int filter_factor, int n_init, uint64_t seed,
                      int32_t *out_i, double *out_d, int32_t *out_status, double *ms_out);

/* The deterministic core of the above for caller-provided replicates: problem q = K[q] distinct values
 * x[q * kcap ..] with multiplicities counts[q * kcap ..] and n_init forced k-means++ seed pairs
 * init[q * 2 * n_init ..] (indices into x).  out[q] = {mean0, weight0, stdev0, mean1, weight1, stdev1, n_peaks}
 * as fit_gmm + the per-replicate bookkeeping of call_alleles (allele.py:249-293) produce them. */
int strk_gmm_fit_counts(strk_ctx *ctx, const double *x, const int32_t *counts, const int32_t *K, const int32_t *init,
                        int64_t n_problems, int kcap, int n_alleles, int num_bootstrap, int min_allele_reads,
                        int force_gm_filter, double expansion_ratio, int filter_factor, int n_init, double *out);

/*
 * The same for per-locus allele counts (STRkitLocus.n_alleles, from the ploidy config): n_alleles[l] in 1..8, one
 * batch for any mix.  Rows have S = the largest count of the batch as their stride:
 *   out_i[l]       1 + 5 * S ints: modal_n, call[S], call_95_cis[S][2], call_99_cis[S][2]
 *   out_d[l]       3 * S doubles: means[S], weights[S], stdevs[S]
 * locus l fills the first n_alleles[l] columns of each group and the rest are 0.
 *   out_status[l]  0, 1, 2 as above, and 3 = at least min_reads reads and two distinct copy numbers but fewer reads
 *                  than n_alleles[l]: the reference's GaussianMixture(n_components = n_alleles).fit raises
 *                  "Expected n_samples >= n_components" there, so no call is made (the row is 0)
 * Loci with one or two alleles are computed by the same code as in the entry above: with the same seed, and a batch
 * that fits one chunk of replicate scratch, their rows are identical.  Three or more alleles run fit_gmm's staged
 * loop (allele.py:56-123: refits with fewer components while the filters find useless ones, the strict filter
 * 1 / (filter_factor * k) for k > 2) and fill the alleles a replicate has no peak for with components drawn by weight
 * (:249-293).  An n_alleles outside 1..8 is STRK_ERR_UNSUPPORTED, and the message names the locus.
 */
int strk_call_alleles_ploidy(strk_ctx *ctx, const int32_t *cn, const double *weights, const int64_t *read_begin,
                             int64_t n_loci, const int32_t *n_alleles, int num_bootstrap, int min_reads,
                             int min_allele_reads, int force_gm_filter, double expansion_ratio, int filter_factor,
                             int n_init, uint64_t seed, int32_t *out_i, double *out_d, int32_t *out_status,
                             double *ms_out);

/* The deterministic core of the above for caller-provided replicates with their own allele counts n_alleles[q]
 * (1..8): problem q = K[q] distinct values x[q * kcap ..] with multiplicities counts[q * kcap ..] (at least
 * n_alleles[q] points when two or more values are present).  init (NULL = k-means++ from a Philox stream keyed by
 * seed and q) holds the forced seeds of every fit the staged loop may run: for nc = A, A-1, ..., 2, n_init rows of nc
 * indices into x; problems follow each other, n_init * (A * (A + 1) / 2 - 1) entries for a problem with A alleles.
 * out[q] has 3 * S + 1 doubles (S = the largest n_alleles): means[S], weights[S], stdevs[S], n_peaks; the first A of
 * each group are sorted by mean, the rest are 0; n_peaks is the fitted component count.  When n_peaks < A the other
 * A - n_peaks entries are copies of fitted components drawn at random by weight, so only the fitted part is
 * deterministic; a forced problem makes no other random draw. */
int strk_gmm_fit_counts_ploidy(strk_ctx *ctx, const double *x, const int32_t *counts, const int32_t *K,
                               const int32_t *n_alleles, const int32_t *init, int64_t n_problems, int kcap,
                               int num_bootstrap, int min_allele_reads, int force_gm_filter, double expansion_ratio,
                               int filter_factor, int n_init, uint64_t seed, double *out);

/* strk_gmm_fit_counts_ploidy through the warp-cooperative fit of deep loci, for K[q] up to kcap <= 4096 and any
 * number of points: one warp per problem, k-means++ and EM over its nonzero (value, count) pairs with warp reductions
 * (the same arithmetic per pair, sums in another order), fit_gmm's staged loop and the fill as above.  Same arguments
 * and output; the k-means++ stream (init NULL) is keyed by seed and q but differs from the per-thread entry's. */
int strk_gmm_fit_counts_deep(strk_ctx *ctx, const double *x, const int32_t *counts, const int32_t *K,
                             const int32_t *n_alleles, const int32_t *init, int64_t n_problems, int kcap,
                             int num_bootstrap, int min_allele_reads, int force_gm_filter, double expansion_ratio,
                             int filter_factor, int n_init, uint64_t seed, double *out);

/* The aggregation step alone (allele.py:295-336): replicate arrays [locus][allele][replicate] (+ peaks
 * [locus][replicate]) -> out_i / out_d as in strk_call_alleles, for n_alleles 1..8. */
int strk_alleles_aggregate(strk_ctx *ctx, const double *rep_means, const double *rep_weights, const double *rep_stdevs,
                           const uint8_t *rep_peaks, int64_t n_loci, int n_alleles, int num_bootstrap, int32_t *out_i,
                           double *out_d);

/*
 * Soft-clip realignment (strkit/call/realign.py:34-72): parasail.sg_dx_trace_scan_16(ref_seq, query_seq, 7, 0,
 * dna_matrix) for n (reference window, read) pairs -- the window aligned end to end, both read ends free, affine gaps
 * (a gap of length k costs gap_open + (k - 1) * gap_extend; the reference passes 7 and 0), traceback.
 *   ref_off / ref_len, read_off / read_len   ASCII sequences in `arena`
 *   score[k], end_ref[k]    parasail's result fields (end_ref = 0-based last read position aligned)
 *   cigar + cigar_off[k]    the CIGAR from cell (0, 0) in parasail's / BAM's encoding, (len << 4) | op with I = 1 (window
 *                           base against nothing), D = 2 (read base against nothing), '=' = 7, X = 8; the caller sizes
 *                           each region (cigar_off has n + 1 entries) to at least 2 * ref_len + 4 entries
 *   cigar_len[k]            entries written
 * trace_flags: STRK_TRACE_* tie rules of the traceback that the reference tree cannot show (0 = extend on an
 * open / extend tie, diagonal before horizontal before vertical, first best end column).  One byte of device memory
 * per DP cell while a group of alignments is in flight (groups are cut at STRK_REALIGN_TRACE_MB, default 2048).
 */
#define STRK_TRACE_OPEN_ON_TIE 1
#define STRK_TRACE_INS_FIRST 2
#define STRK_TRACE_END_LAST 4
int strk_realign(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *ref_off, const int32_t *ref_len,
                 const uint64_t *read_off, const int32_t *read_len, int64_t n, int gap_open, int gap_extend, int trace_flags,
                 int32_t *score, int32_t *end_ref, uint32_t *cigar, const uint64_t *cigar_off, int32_t *cigar_len);

/* Integer issue-rate micro-benchmark: the roofline denominator of the DP kernels (MEASURED_PEAKS.json has
 * no INT32 figure).  out_tiops[0] = ALU pipe only (VIADDMNMX), [1] = FMA pipe only (IMAD), [2] = both pipes;
 * units: 1e12 lane-level 32-bit integer instructions per second, all SMs. */
int strk_measure_int_peak(strk_ctx *ctx, double out_tiops[3]);

#ifdef __cplusplus
}
#endif
#endif
