/*
 * kmerml_b200.h -- C-ABI of libkmerml_b200.so: the B200 (sm_100a) implementation of
 * kmer-ml's k-mer extraction -> counts -> feature-matrix hot path.
 *
 * The reference (Masthetheus/kmer-ml) is pure Python and has no FFI; this header is
 * the boundary a maintainer would bind with ctypes (see INTEGRATION.md).  Each entry
 * point names the reference code it replaces (paths relative to the reference tree).
 *
 * Conventions
 *   - every function returns an int status: KMERML_OK or a negative KMERML_ERR_*;
 *     nothing throws or aborts; kmerml_last_error() gives the thread-local message;
 *   - plain pointers and sizes only; "d_" pointers are device memory of the context's
 *     GPU (16-byte aligned), "h_" pointers are host memory (pinned for full speed);
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream);
 *     device entry points are asynchronous on it, *_host entry points synchronise;
 *     a context's scratch memory is shared by its calls, so a call on another stream than
 *     the context's previous call first waits (on the device) for that call to finish;
 *   - k-mer index = lexicographic ACGT (A0 C1 G2 T3), first base most significant;
 *     the on-disk digit code A0 T1 C2 G3 (kmerml/kmers/generate.py:71) is applied
 *     only by the text writer;
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef KMERML_B200_H
#define KMERML_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMERML_OK 0
#define KMERML_ERR_ARG (-1)     /* bad argument */
#define KMERML_ERR_CUDA (-2)    /* CUDA runtime error (message has the details) */
#define KMERML_ERR_NOMEM (-3)   /* host or device allocation failed */
#define KMERML_ERR_RANGE (-4)   /* input too large for the 32-bit counters / offsets */

#define KMERML_FLAG_CANONICAL 1u /* count min(kmer, revcomp) -- opt-in extension, not in the reference */
#define KMERML_FLAG_K8_AS_9 8u      /* k = 8: count 9-mers through the partition path instead of the packed shared histogram */
#define KMERML_FLAG_NO_PARTITION 2u /* k = 9..12: use the global-atomic kernel instead of the partition path */

#define KMERML_MAX_DENSE_K 14    /* dense 4^k histograms up to here; larger k -> kmerml_count_sparse */
#define KMERML_MAX_K 32
#define KMERML_N_STATIC_FEATURES 14

typedef struct kmerml_ctx kmerml_ctx;

int kmerml_version(void);
const char *kmerml_last_error(void);

/*
 * One context per GPU per host thread.  Owns scratch/staging memory and streams.
 * Environment: KMERML_GROUP_PAYLOAD_MB=<n> (read by kmerml_ctx_create) bounds the partition workspace one
 * group of genomes may take (default 12288); smaller values trade workspace for more kernel launches.
 */
int kmerml_ctx_create(int device, kmerml_ctx **out);
int kmerml_ctx_destroy(kmerml_ctx *ctx);
int kmerml_ctx_sm_count(const kmerml_ctx *ctx);

/* Elements in one output row: sum over k_list of 4^k. */
uint64_t kmerml_row_len(const int *k_list, int nk);

/*
 * Dense k-mer counting of a batch of genomes that is already resident in HBM.
 * Replaces kmerml/kmers/generate.py:36-58 (KmerExtractor.extract_kmers_from_fasta:
 * record loop :39, upper-casing :41, short-record skip :44-46, window loop :49-52,
 * ACGT filter :55-56, count :58) for every k in k_list (all <= KMERML_MAX_DENSE_K),
 * and adds the per-genome frequency row (count / windows) the reference only
 * gestures at (tests/test_ml.py:8 normalize(method="frequency")).
 *
 *   d_fasta      raw FASTA file bytes of all genomes, concatenated back to back
 *   h_offsets    n_genomes+1 byte offsets into d_fasta (genome g = [off[g], off[g+1]))
 *   k_list       distinct k values, any order (output row follows this order)
 *   min_record_len  records shorter than this contribute nothing (the reference uses
 *                max(k_values) over ALL requested k, generate.py:44); 0 = max(k_list)
 *   d_counts     [n_genomes][counts_stride] uint32, row g = concat_k counts_k[4^k]
 *   d_freq       same shape in float32, or NULL
 *   d_totals     [n_genomes][nk] uint64 counted windows per k, or NULL
 */
int kmerml_count_dense_batch(kmerml_ctx *ctx, const uint8_t *d_fasta, const uint64_t *h_offsets,
                             int n_genomes, const int *k_list, int nk, int min_record_len,
                             unsigned flags, uint32_t *d_counts, uint64_t counts_stride,
                             float *d_freq, uint64_t freq_stride, uint64_t *d_totals,
                             void *stream);

/*
 * One genome, only the windows whose LAST base lies in bytes [range_begin, range_end) of the
 * file: the unit of intra-genome parallelism.  Ranges that tile the file give partial count
 * rows (all requested k, cascade included) and partial window totals whose SUM over the ranges
 * is exactly the whole-genome result -- across GPUs that sum is one NCCL all-reduce of
 * uint32[row_len] (SURVEY 8e).  The k-1 bases before range_begin are read from the file itself,
 * so no overlap bookkeeping is needed.  range_begin must be a multiple of 16384; no frequencies
 * are written (normalise after the reduction with kmerml_normalize_rows).
 */
int kmerml_count_dense_range(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes,
                             uint64_t range_begin, uint64_t range_end, const int *k_list, int nk,
                             int min_record_len, unsigned flags, uint32_t *d_counts,
                             uint64_t *d_totals, void *stream);

/*
 * The same path end to end from HOST buffers: per genome H2D copy -> counting ->
 * D2H of the counts and totals, pipelined over three device slots.  h_counts / h_totals
 * are laid out like their d_ counterparts.  The frequency rows go where the caller needs
 * them: `freq` is a HOST buffer (copied back like the counts) or, with
 * KMERML_FLAG_FREQ_ON_DEVICE, a DEVICE buffer [n_genomes][freq_stride] that keeps the
 * feature matrix resident in HBM for the distance / ML stage; NULL = not computed.
 * Synchronous.
 */
#define KMERML_FLAG_FREQ_ON_DEVICE 4u
/* By default the count rows of k >= 10 cross PCIe as one byte per bin plus an exception list and are widened to
 * uint32 in the caller's buffer by host threads (KMERML_HOST_THREADS, default half the cores, at most 16) while
 * the next genomes are in flight; lossless.  This flag copies the uint32 rows as they are instead. */
#define KMERML_FLAG_WIDE_D2H 16u
/* ... and a level of k >= 10 whose mean count is at most 5 (genome bytes <= 5 * 4^k) even as FOUR BITS per bin (bins
 * that reached 15 go to the exception list).  This flag keeps every level at one byte per bin. */
#define KMERML_FLAG_NO_NIBBLES 32u
/* Number of host threads that widen the narrow format (one process per GPU: cores / ranks on the host). */
int kmerml_ctx_set_host_threads(kmerml_ctx *ctx, int n_threads);
int kmerml_count_dense_host(kmerml_ctx *ctx, const uint8_t *const *h_fasta, const uint64_t *h_sizes,
                            int n_genomes, const int *k_list, int nk, int min_record_len,
                            unsigned flags, uint32_t *h_counts, uint64_t counts_stride,
                            float *freq, uint64_t freq_stride, uint64_t *h_totals);

/*
 * The same call with the result left in the form it crosses PCIe in: per genome one row of
 * kmerml_compact_row_bytes(k_list, nk) bytes (stride a multiple of 16):
 *     [ header: "KMW2", bit mask of the k_list entries packed as nibbles, 8 bytes reserved |
 *       one byte -- or one nibble, low one first -- per bin of every k >= 10, in k_list order |
 *       exception count (uint32, padded to 16 bytes) | 32768 x (row-relative bin, count) uint32 pairs for the bins
 *       that reached 255 (15 in a nibble level) | the uint32 rows of every k < 10, in k_list order ]
 * Lossless unless the exception count exceeds 32768 (kmerml_compact_row_overflowed / kmerml_compact_expand report it;
 * count that genome with kmerml_count_dense_host).  Four to six times fewer bytes
 * cross the bus and none is rewritten by the host; kmerml_compact_expand widens one k of one genome on demand
 * (pure host code, no GPU).  The host memory of this pool's boxes takes writes at ~60 GB/s, which is what bounds
 * the uint32 variant above.
 */
uint64_t kmerml_compact_row_bytes(const int *k_list, int nk);
int kmerml_count_dense_host_compact(kmerml_ctx *ctx, const uint8_t *const *h_fasta, const uint64_t *h_sizes,
                                    int n_genomes, const int *k_list, int nk, int min_record_len,
                                    unsigned flags, uint8_t *h_rows, uint64_t row_stride_bytes, float *freq,
                                    uint64_t freq_stride, uint64_t *h_totals);
int kmerml_compact_expand(const int *k_list, int nk, const uint8_t *h_row, int ki, uint32_t *h_out);
int kmerml_compact_row_overflowed(const int *k_list, int nk, const uint8_t *h_row);   /* 1 / 0, negative: error */
uint64_t kmerml_compact_row_used_bytes(const int *k_list, int nk, const uint8_t *h_row);   /* bytes that crossed the bus */

/*
 * Sparse counting for 15 <= k <= 32 (any k >= 1 is accepted): the distinct k-mers of ONE genome as
 * sorted 2-bit packed keys (A0 C1 G2 T3, first base most significant), their counts, and the byte
 * offset of the last base of each k-mer's first window (sort by it for dict insertion order,
 * generate.py:88).  Same window rules as the dense path.  Synchronous.  *h_unique receives the
 * number of distinct k-mers; when it exceeds out_cap nothing is written: call again with larger
 * outputs.  Genome < 4 GiB.  d_first may be NULL.
 */
int kmerml_count_sparse(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, int k, int min_record_len,
                        unsigned flags, uint64_t *d_keys, uint32_t *d_counts, uint32_t *d_first,
                        uint64_t out_cap, uint64_t *h_unique, uint64_t *h_windows, void *stream);

/*
 * The result of the last kmerml_count_sparse / kmerml_count_sparse_range call of this context whose
 * *h_unique exceeded out_cap, copied out of the workspace without counting again (out_cap >= that number;
 * no other call may have used the context in between).  Synchronous.
 */
int kmerml_sparse_fetch(kmerml_ctx *ctx, uint64_t *d_keys, uint32_t *d_counts, uint32_t *d_first,
                        uint64_t out_cap, void *stream);

/*
 * Multi-GPU unit of the sparse path (SURVEY 8e, "one large genome, sparse k"): the same as
 * kmerml_count_sparse for the windows whose last base lies in the byte range [range_begin, range_end) of
 * the file -- begin a multiple of KMERML_SPARSE_RANGE_ALIGN, end too or == nbytes.  The k-1 bases before
 * the range are read from the file itself, so the ranges of all ranks tile the genome without overlap
 * bookkeeping; first offsets are relative to the file, not to the range.
 */
#define KMERML_SPARSE_RANGE_ALIGN 131072
int kmerml_count_sparse_range(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, uint64_t range_begin,
                              uint64_t range_end, int k, int min_record_len, unsigned flags, uint64_t *d_keys,
                              uint32_t *d_counts, uint32_t *d_first, uint64_t out_cap, uint64_t *h_unique,
                              uint64_t *h_windows, void *stream);

/*
 * Merge of partial sparse results (what a rank holds after the all-to-all that routes every k-mer to
 * the rank owning its key range): n (k-mer, count, first) triples in any order, duplicates allowed ->
 * distinct k-mers ascending, counts added, smallest first offset kept.  d_first / d_first_out may be
 * NULL.  *h_unique always receives the number of distinct k-mers; when it exceeds out_cap nothing is
 * written.  Synchronises `stream`.
 */
int kmerml_merge_sparse(kmerml_ctx *ctx, int k, const uint64_t *d_keys, const uint32_t *d_counts,
                        const uint32_t *d_first, uint64_t n, uint64_t *d_keys_out, uint32_t *d_counts_out,
                        uint32_t *d_first_out, uint64_t out_cap, uint64_t *h_unique, void *stream);

/*
 * Multi-GPU units of the sparse path with RAW routing (each rank sorts once): kmerml_emit_sparse_range emits the windows
 * of a byte range -- 2-bit packed k-mer (canonical with the flag) and the byte offset of its last base -- grouped by the
 * rank that owns them: owner = the top owner_bits bits of the 2k-bit k-mer (2^owner_bits ranks; one radix pass);
 * h_owner_counts[2^owner_bits] receives the group sizes, *h_windows their sum (nothing is written when it exceeds
 * out_cap; at most one window ends at every byte of the range).  After the all-to-all every rank calls
 * kmerml_reduce_sparse_windows on what it received: one radix sort over the low sort_bits bits (2k - owner_bits: the
 * owner bits are equal on a rank) + one fused segmented reduction -> distinct k-mers ascending, counts, smallest
 * offset; *h_unique > out_cap: fetch with kmerml_sparse_fetch.  Both synchronous.
 */
int kmerml_emit_sparse_range(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, uint64_t range_begin,
                             uint64_t range_end, int k, int min_record_len, unsigned flags, int owner_bits,
                             uint64_t *d_keys, uint32_t *d_ends, uint64_t out_cap, uint64_t *h_windows,
                             uint64_t *h_owner_counts, void *stream);
int kmerml_reduce_sparse_windows(kmerml_ctx *ctx, int sort_bits, const uint64_t *d_keys, const uint32_t *d_ends,
                                 uint64_t n, uint64_t *d_keys_out, uint32_t *d_counts_out, uint32_t *d_first_out,
                                 uint64_t out_cap, uint64_t *h_unique, void *stream);

/*
 * Byte offset (within the genome) of the last base of the first window of every
 * k-mer, UINT32_MAX where the k-mer never occurs: sorting the observed bins by
 * this value gives dict insertion order, i.e. the line order of k{k}.txt
 * (kmerml/kmers/generate.py:88).  One genome, one k (<= KMERML_MAX_DENSE_K),
 * genome smaller than 4 GiB.  d_first: uint32[4^k].
 */
int kmerml_first_occurrence(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, int k,
                            int min_record_len, uint32_t *d_first, void *stream);

/*
 * Text of a k{k}.txt file from a dense count row: one line "<digits>\t<count>\n" per observed k-mer
 * (digits A0 T1 C2 G3), lines in order of first occurrence -- the writer of
 * kmerml/kmers/generate.py:68-91.  d_counts: uint32[4^k], one genome's row of one k
 * (kmerml_count_dense_batch); d_first: kmerml_first_occurrence's output for the same genome, k and
 * min_record_len.  KMERML_FLAG_CANONICAL: d_counts is a canonical row.  max_lines bounds the observed
 * k-mers and text_cap the bytes of d_text; *h_lines / *h_text_len always receive the real numbers, and
 * when one exceeds its bound nothing is written: re-size and call again.  Synchronises `stream`.
 */
int kmerml_format_kmer_file(kmerml_ctx *ctx, int k, const uint32_t *d_counts, const uint32_t *d_first,
                            unsigned flags, uint64_t max_lines, uint8_t *d_text, uint64_t text_cap,
                            uint64_t *h_text_len, uint64_t *h_lines, void *stream);

/*
 * The same text from k-mers that are already in line order (kmerml_count_sparse's output sorted by
 * first occurrence): d_codes uint64[n] 2-bit packed (A0 C1 G2 T3), d_counts uint32[n], k <= 32.
 */
int kmerml_format_kmer_lines(kmerml_ctx *ctx, int k, const uint64_t *d_codes, const uint32_t *d_counts,
                             uint64_t n, uint8_t *d_text, uint64_t text_cap, uint64_t *h_text_len, void *stream);

/*
 * Record table of one FASTA file resident in HBM: byte offsets of the header lines
 * (unordered; sort them) -- what Bio.SeqIO.parse would yield one record for
 * (kmerml/kmers/generate.py:39).  *h_count receives the number found (may exceed cap;
 * then call again with a larger buffer).  Synchronous.
 */
int kmerml_find_records(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, uint64_t *d_offsets,
                        uint32_t cap, uint32_t *h_count, void *stream);
/*
 * For n records given by the (sorted or not) header offsets: is_short[i] = 1 when the
 * record holds fewer than min_record_len symbols -- the records generate.py:44-46 skips
 * with "Skipping <id>: too short for k-mer extraction".
 */
int kmerml_records_short(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, const uint64_t *d_offsets,
                         uint32_t n, int min_record_len, uint8_t *d_is_short, void *stream);

/*
 * Genome tallies of one FASTA file resident in HBM, as kmerml/utils/genome_metadata.py:55-85 computes
 * them: d_out[0] contigs (records), [1] total_size (symbols of all records), [2] G+C count,
 * [3] N count (either case).  Asynchronous on `stream`; d_out: uint64[4] device memory.
 */
int kmerml_genome_stats(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, uint64_t *d_out, void *stream);

/*
 * The exchange step of the chunked single-genome path (SURVEY 8b / 8e row 2) for hosts that drive NCCL themselves:
 * sums a count row over the ranks of `nccl_comm` (a ncclComm_t passed as void*), in place, on `stream`.
 *   reduce_scatter = 0: all-reduce -- every rank ends with the whole row;
 *   reduce_scatter = 1: rank r ends with slice r, n / nranks elements at d_counts + r * (n / nranks)
 *                       (n must divide evenly); the other slices of its buffer are left as they were.
 * dtype: 0 = uint32, 1 = uint64.  Integer sums: bit-identical to counting the whole genome on one GPU.
 * NCCL is taken from the calling process at run time (dlopen of libnccl.so.2 -- the one torch or the host
 * application already loaded); this library does not link it, and the call fails with KMERML_ERR_ARG when there
 * is none.  (kmerml_b200/dist.py makes the same exchange through torch.distributed.)
 */
int kmerml_allreduce_counts(kmerml_ctx *ctx, void *nccl_comm, void *d_counts, uint64_t n, int dtype,
                            int reduce_scatter, void *stream);

/*
 * Stage 1 on its own (SURVEY 8b `kmerml_encode`): the symbols of one FASTA file resident in HBM, as the counting
 * kernels see them after kmerml/kmers/generate.py:39-41,55-56 -- d_symbols[i] = 0..3 (A C G T, either case) when
 * byte i is a base of a record, 0xFF for everything else (header lines, line ends, N / IUPAC codes, blanks, text
 * before the first '>').  d_tallies (uint64[4], may be NULL) receives the tallies of kmerml_genome_stats.
 * The counting entry points do NOT need this: they decode in registers; it is for callers that want the symbol
 * stream itself.  Asynchronous on `stream`.
 */
int kmerml_encode(kmerml_ctx *ctx, const uint8_t *d_fasta, uint64_t nbytes, uint8_t *d_symbols, uint64_t *d_tallies,
                  void *stream);

/*
 * Static per-k-mer features (functions of the k-mer string only): replaces the per-row
 * helpers of kmerml/kmers/statistics.py:190-240.  d_out: int32[4^k][8] =
 * {n, A_count, C_count, G_count, T_count, cpg_count, has_repeat, first base}, row index =
 * lexicographic ACGT k-mer index.  compat != 0 computes them on the string the reference's
 * CSV actually holds (leading 'A's lost to pandas' integer parsing, statistics.py:261-271).
 * The float columns (gc_percent, cpg_obs_exp, entropies) are pure functions of these
 * integers and are derived by the host with the reference's own float expressions.
 */
int kmerml_static_features(kmerml_ctx *ctx, int k, int compat, int32_t *d_out, void *stream);

/* out[g][i] = counts[g][i] / totals[g] (float32): frequency normalisation of count rows. */
int kmerml_normalize_rows(kmerml_ctx *ctx, const uint32_t *d_counts, uint64_t counts_stride,
                          const uint64_t *d_totals, int n_rows, uint64_t m, float *d_out,
                          uint64_t out_stride, void *stream);

/*
 * Genome x genome distance matrix of the rows of X (n x m): metric 0 = cosine,
 * 1 = Euclidean.  dtype 0 = float32, 1 = uint32 (count rows: the Gram matrix is then
 * exact), 2 = float64.  Accumulation is float64 (the north star's 1e-6 relative
 * tolerance).  d_out32 / d_out64: n x n, either may be NULL.  uint32 rows with m a multiple of 64 go to the
 * tensor cores, for m up to 65535 x 32768 features (every concatenated dense row fits; longer: KMERML_ERR_RANGE).
 */
#define KMERML_METRIC_COSINE 0
#define KMERML_METRIC_EUCLIDEAN 1
int kmerml_pairwise_distance(kmerml_ctx *ctx, const void *d_x, int dtype, uint64_t stride, int n,
                             uint64_t m, int metric, float *d_out32, double *d_out64, void *stream);

/*
 * The per-k-mer feature CSV of kmerml/kmers/statistics.py:95-251 as text produced on the GPU (featcsv.cu).
 *   kmerml_parse_kmer_lines      the lines "<digits>\t<count>" of a k{k}.txt image in HBM -> int64 value (leading
 *                                zeros lost, as pandas reads the column, :261-271) and count; d_line_end[i] = byte
 *                                offset of the terminator of line i; *h_bad != 0: some line is not of that form (or
 *                                has more than 18 digits): the caller takes the reference's pandas path.  Synchronous.
 *   kmerml_feature_keys          composition class of str(value) decoded 0 A 1 T 2 C 3 G else N (:248-251):
 *                                length | A << 5 | C << 10 | G << 15 | T << 20 | N << 25 | CpG count << 30 | repeat << 35;
 *                                every feature column of :149-240 is a function of it
 *   kmerml_feature_line_lengths  bytes of "<letters>,<count>,<suffix>\n" per row (suffix = the class's formatted columns)
 *   kmerml_feature_write_lines   those lines at the given offsets (exclusive prefix sums of the lengths)
 */
int kmerml_parse_kmer_lines(kmerml_ctx *ctx, const uint8_t *d_text, const int64_t *d_line_end, uint64_t n_lines,
                            int64_t *d_value, int64_t *d_count, uint32_t *h_bad, void *stream);
int kmerml_feature_keys(kmerml_ctx *ctx, const int64_t *d_value, uint64_t n_rows, int64_t *d_keys, void *stream);
int kmerml_feature_line_lengths(kmerml_ctx *ctx, const int64_t *d_value, const int64_t *d_count,
                                const int64_t *d_class, const int32_t *d_suffix_len, uint64_t n_rows,
                                int64_t *d_len, void *stream);
int kmerml_feature_write_lines(kmerml_ctx *ctx, const int64_t *d_value, const int64_t *d_count,
                               const int64_t *d_class, const int64_t *d_suffix_off, const int32_t *d_suffix_len,
                               const uint8_t *d_suffix_text, const int64_t *d_line_off, uint64_t n_rows,
                               uint8_t *d_out, void *stream);

/*
 * Summary of one k's count row as kmerml/utils/kmer_metadata.py:59-78 reports it for a k{k}.txt file (the
 * OBSERVED k-mers only): d_out uint64[8] = total_kmers, unique_kmers, max_count, min_count, the lower and the
 * upper middle count (their mean is the median; equal for an odd number), 0, 0.  No observed k-mer: total =
 * unique = max = 0, min = 2^64 - 1.  The median is an exact three-pass radix select, not a sort.
 */
int kmerml_count_stats(kmerml_ctx *ctx, const uint32_t *d_counts, uint64_t n_bins, uint64_t *d_out, void *stream);

/*
 * Per column of an n_rows x m feature matrix (dtype as in kmerml_pairwise_distance): rows with a non-zero entry,
 * mean and population variance in float64 -- the reductions behind filter_features(min_prevalence, min_variance)
 * and get_top_features(n, "variance"), the calls tests/test_ml.py:9-12 of the reference makes to methods its
 * kmerml/ml/features.py does not define.
 */
int kmerml_column_stats(kmerml_ctx *ctx, const void *d_x, int dtype, uint64_t stride, int n_rows, uint64_t m,
                        uint32_t *d_nnz, double *d_mean, double *d_var, void *stream);

/*
 * Rows [row_begin, row_end) of that matrix for uint32 count rows (m a multiple of 64): the block one
 * GPU computes when the genomes were counted on several GPUs and the rows gathered (the reference has no
 * distance code; nearest hooks are the stubs kmerml/ml/clustering.py:6-16).  All n rows must be resident;
 * d_out32 / d_out64: (row_end - row_begin) x n.  The Gram entries are exact integers (tcgen05 kind::i8), so
 * the block is bit-identical to the same rows of kmerml_pairwise_distance.  m up to 65535 x 32768 features, as there
 * (longer: KMERML_ERR_RANGE).
 */
int kmerml_pairwise_distance_rows(kmerml_ctx *ctx, const uint32_t *d_counts, uint64_t stride, int n,
                                  uint64_t m, int row_begin, int row_end, int metric, float *d_out32,
                                  double *d_out64, void *stream);

/*
 * The same in two steps, for genomes counted on several GPUs (SURVEY 8e row 1): every rank turns ITS count rows into
 * byte planes, the planes -- one byte per bin and plane, not the uint32 rows -- are gathered, and every rank computes
 * its row block from the planes of all rows.
 *   kmerml_count_planes: plane d (d = 0..3, at d_planes + d * plane_stride, n x m bytes) = byte d of every count;
 *     d_sumsq[row] (may be NULL) = the row's exact squared norm; *d_max (device, zeroed by the caller) = atomicMax
 *     of the counts: planes 0 .. (bytes needed for the largest count of ALL ranks) - 1 are the ones to gather.
 *   kmerml_distance_rows_planes: rows [row_begin, row_end) of the n x n matrix from n_planes planes of all n rows
 *     and their squared norms; rows of zeros (padding) are allowed.  Bit-identical to kmerml_pairwise_distance.
 */
int kmerml_count_planes(kmerml_ctx *ctx, const uint32_t *d_counts, uint64_t stride, int n, uint64_t m, uint8_t *d_planes,
                        uint64_t plane_stride, double *d_sumsq, uint32_t *d_max, void *stream);
int kmerml_distance_rows_planes(kmerml_ctx *ctx, const uint8_t *d_planes, uint64_t plane_stride, int n_planes, int n,
                                uint64_t m, const double *d_sumsq, int row_begin, int row_end, int metric,
                                float *d_out32, double *d_out64, void *stream);

/*
 * MinHash genome sketches and their Mash / Jaccard distances, for any k up to 32 (Ondov et al. 2016).
 *
 * kmerml_sketch_batch: the bottom-s sketch of every genome of a batch laid out as for kmerml_count_dense_batch
 * (genome g = bytes [h_offsets[g], h_offsets[g + 1]) of d_fasta, 16-byte aligned).  k-mer keys and window rules are
 * those of kmerml_count_sparse (KMERML_FLAG_CANONICAL: min(forward, reverse complement); min_record_len 0 means k).
 * A key is hashed as h = fmix64(key + 0x9E3779B97F4A7C15 * (seed + 1)) mod 2^64 (fmix64: MurmurHash3's 64-bit
 * finalizer), a bijection, so distinct hashes are distinct k-mers.  The sketch of genome g is the min(s, D) smallest
 * distinct hashes of its k-mers (D = its distinct k-mers), ascending, in d_sketches[g * sketch_stride ..]; slots past
 * d_filled[g] = min(s, D) hold UINT64_MAX.  These sketches are not file-compatible with Mash or sourmash.
 * Every window is hashed once per round; only those below a per-genome threshold (~3 s of them) are stored.  A genome
 * with fewer than s distinct hashes below its threshold, or whose stored windows overflowed their region (tandem
 * repeats of a low-hash k-mer), is run again with a larger threshold or region, up to "keep every window".
 * 1 <= s <= KMERML_SKETCH_MAX, sketch_stride >= s.  Synchronous.
 *
 * kmerml_sketch_distance_rows: rows [row_begin, row_end) x all n columns of the distance matrix of n sketches of
 * kmerml_sketch_batch (same k, s, seed and canonical flag).  For sketches A and B: U = the min(s, |A u B|) smallest
 * values of A u B, x = |U n A n B|, j = x / |U| (0 when |U| = 0); KMERML_SKETCH_METRIC_JACCARD gives 1 - j,
 * KMERML_SKETCH_METRIC_MASH gives -ln(2j / (1 + j)) / k (1 when j = 0, 0 when j = 1).  Computed in float64;
 * d_out32 / d_out64 ((row_end - row_begin) x n, either may be NULL) receive that value (rounded for float32).  The
 * matrix is exactly symmetric, and a row block is bit-identical to the same rows of the whole matrix.
 */
#define KMERML_SKETCH_MAX 16384
#define KMERML_SKETCH_METRIC_MASH 0
#define KMERML_SKETCH_METRIC_JACCARD 1
int kmerml_sketch_batch(kmerml_ctx *ctx, const uint8_t *d_fasta, const uint64_t *h_offsets, int n_genomes,
                        int k, int min_record_len, unsigned flags, int sketch_size, uint64_t seed,
                        uint64_t *d_sketches, uint64_t sketch_stride, uint32_t *d_filled, void *stream);
int kmerml_sketch_distance_rows(kmerml_ctx *ctx, const uint64_t *d_sketches, uint64_t sketch_stride,
                                const uint32_t *d_filled, int n, int sketch_size, int k, int row_begin, int row_end,
                                int metric, float *d_out32, double *d_out64, void *stream);

/*
 * Scaled (FracMinHash) genome sketches and their containment, Jaccard and containment ANI, for any k up to 32
 * (Irber et al. 2022; containment ANI: Hera et al. 2023).  Unlike a bottom-s sketch, a scaled sketch grows with the
 * genome, so a small genome (a plasmid, a MAG) can be compared with a large one by containment.
 *
 * kmerml_fmh_batch: the scaled sketch of every genome of a batch laid out as for kmerml_sketch_batch, with the same
 * keys, window rules, KMERML_FLAG_CANONICAL, min_record_len (0 means k) and hash h = fmix64(key + 0x9E3779B97F4A7C15 *
 * (seed + 1)).  The sketch of genome g is every distinct hash h <= T = floor((2^64 - 1) / scale) of its k-mers,
 * ascending (scale 1: every distinct k-mer).  With equal k, seed and canonical flag, its first s values are the
 * bottom-s sketch of kmerml_sketch_batch whenever it holds at least s values.  The sketches come out in genome order
 * as CSR: genome g is d_hashes[off[g] .. off[g + 1]), off = d_sketch_offsets (n_genomes + 1 values, always written).
 * *h_total always receives off[n_genomes]; when it exceeds out_cap the hashes are not written: call
 * kmerml_fmh_fetch with outputs that large.  Every window is hashed once; the windows at or below T are stored in a
 * region of about twice the expected count per genome, and a genome whose region overflowed (tandem repeats of a
 * low-hash k-mer) runs again with a region of exactly its stored windows.  A genome whose windows at or below T
 * exceed 2^31 - 1 returns KMERML_ERR_RANGE (scale 1 on a genome of more than 2 Gbp: use a larger scale).
 * scale >= 1.  Synchronous.
 *
 * kmerml_fmh_fetch: the result of the last kmerml_fmh_batch call of this context, copied out of the context without
 * walking the FASTA again (out_cap >= its total).  Later calls of other functions do not disturb it.  Synchronous.
 *
 * kmerml_fmh_compare: for every query q < n_q and reference r < n_r (two CSR sets of sketches of kmerml_fmh_batch,
 * made with the same k, scale, seed and canonical flag -- not checked here; the two sets may be the same pointers),
 * x = |Q n R| exactly, and the metric in float64 from x, |Q| and |R|: KMERML_FMH_CONTAINMENT x / |Q|,
 * KMERML_FMH_MAX_CONTAINMENT x / min(|Q|, |R|), KMERML_FMH_JACCARD x / (|Q| + |R| - x), KMERML_FMH_CONTAINMENT_ANI
 * (x / |Q|)^(1/k), KMERML_FMH_MAX_CONTAINMENT_ANI (x / min(|Q|, |R|))^(1/k); 0 when x = 0 (so also when a
 * denominator is 0).  All are similarities.  Row q, column r of d_intersections (uint32), d_out32 and d_out64
 * (n_q x n_r each, any of them NULL, not all three) receive x and the metric (rounded for float32).  Asynchronous on
 * `stream`; the result of one query does not depend on the others, so a block of query rows is bit-identical to
 * the same rows of the whole matrix.
 */
#define KMERML_FMH_CONTAINMENT 0
#define KMERML_FMH_MAX_CONTAINMENT 1
#define KMERML_FMH_JACCARD 2
#define KMERML_FMH_CONTAINMENT_ANI 3
#define KMERML_FMH_MAX_CONTAINMENT_ANI 4
int kmerml_fmh_batch(kmerml_ctx *ctx, const uint8_t *d_fasta, const uint64_t *h_offsets, int n_genomes, int k,
                     int min_record_len, unsigned flags, uint64_t scale, uint64_t seed, uint64_t *d_hashes,
                     uint64_t out_cap, uint64_t *d_sketch_offsets, uint64_t *h_total, void *stream);
int kmerml_fmh_fetch(kmerml_ctx *ctx, uint64_t *d_hashes, uint64_t out_cap, uint64_t *d_sketch_offsets, void *stream);
int kmerml_fmh_compare(kmerml_ctx *ctx, const uint64_t *d_q_hashes, const uint64_t *d_q_offsets, int n_q,
                       const uint64_t *d_r_hashes, const uint64_t *d_r_offsets, int n_r, int k, int metric,
                       uint32_t *d_intersections, float *d_out32, double *d_out64, void *stream);

/*
 * k-mer abundance in scaled sketches: how many windows of a genome carry each kept hash, so a metagenome says how much
 * of each genome it holds, not only which genomes.
 *
 * KMERML_FLAG_FMH_ABUNDANCE (flag of kmerml_fmh_batch): also keep, for every value h of every sketch, its abundance
 * a_g(h) = the number of windows of genome g whose key hashes to h (the windows the sketch counts; with
 * KMERML_FLAG_CANONICAL both orientations count toward the canonical key), as uint32.  The stored windows of one genome
 * are at most 2^31 - 1, so every sum below fits uint64 exactly: sum a <= 2^31, sum a_Q a_R <= 2^62, sum a^2 <= 2^62.
 * The hashes and offsets are those of the call without the flag.  Without the flag nothing extra is kept.
 *
 * kmerml_fmh_fetch_abundances: the abundances of the last kmerml_fmh_batch call of this context, in the CSR order of
 * kmerml_fmh_fetch (d_abundances: out_cap >= its total).  KMERML_ERR_ARG when that call was made without
 * KMERML_FLAG_FMH_ABUNDANCE or out_cap is short.  Synchronous.
 *
 * kmerml_fmh_compare_weighted: two CSR sets of sketches as for kmerml_fmh_compare, with their abundances
 * (d_r_abundances may be NULL for KMERML_FMH_WEIGHTED_CONTAINMENT).  For every query q and reference r:
 *   KMERML_FMH_WEIGHTED_CONTAINMENT  x = sum_{h in Q n R} a_Q(h), metric x / sum_{h in Q} a_Q(h): the share of the
 *                                    query's k-mer mass (reads, coverage) that R explains;
 *   KMERML_FMH_ANGULAR_SIMILARITY    x = sum_{h in Q n R} a_Q(h) a_R(h), metric 1 - 2 acos(c) / pi with
 *                                    c = min(1, x / (sqrt(sum_Q a_Q^2) sqrt(sum_R a_R^2))), and c = 1 whenever
 *                                    x^2 = sum_Q a_Q^2 sum_R a_R^2 exactly (proportional abundances, self-similarity).
 * Both are 0 when x = 0 or a denominator is 0.  The integer x goes to d_numerators (uint64), the metric in float64 to
 * d_out64 and rounded to d_out32 (n_q x n_r each, any of them NULL, not all three).  The sums are integers and the
 * product of the two roots commutes, so Q = R gives an exactly symmetric matrix, and a block of query rows is
 * bit-identical to the same rows of the whole matrix.  Asynchronous on `stream`.
 *
 * kmerml_fmh_gather_abundance: kmerml_fmh_gather with the query abundances d_q_abundances (parallel to d_q_hashes).
 * The picks are made on the unweighted counts, so the first outputs are those of kmerml_fmh_gather.  For match t of
 * query q, with S_t the query hashes that match takes, slot q * max_matches + t of d_match_unique_weighted receives
 * sum_{S_t} a_Q (uint64), of d_match_unique_sumsq sum_{S_t} a_Q^2 (uint64), and of d_match_median_abund the median of
 * a_Q over S_t (float64; for an even count the mean of the two middle values, exact).  Extra device workspace:
 * 8 (total query hashes) + 16 n_q bytes and a segmented sort's temporary storage.  Synchronous.
 */
#define KMERML_FLAG_FMH_ABUNDANCE 64u
#define KMERML_FMH_WEIGHTED_CONTAINMENT 5
#define KMERML_FMH_ANGULAR_SIMILARITY 6
int kmerml_fmh_fetch_abundances(kmerml_ctx *ctx, uint32_t *d_abundances, uint64_t out_cap, void *stream);
int kmerml_fmh_compare_weighted(kmerml_ctx *ctx, const uint64_t *d_q_hashes, const uint64_t *d_q_offsets,
                                const uint32_t *d_q_abundances, int n_q, const uint64_t *d_r_hashes,
                                const uint64_t *d_r_offsets, const uint32_t *d_r_abundances, int n_r, int metric,
                                uint64_t *d_numerators, float *d_out32, double *d_out64, void *stream);

/*
 * kmerml_fmh_gather: split each query sketch greedily and exactly into the reference sketches that cover it (gather,
 * Irber et al. 2022: a greedy minimum set cover).  The inputs are two CSR sets of sketches as for kmerml_fmh_compare
 * (same k, scale, seed and canonical flag -- not checked here; the two sets may be the same pointers).  For query Q
 * and references R_0 .. R_{n_r - 1}: Q_0 = Q; in round t = 1, 2, ..., u_t(r) = |Q_{t-1} n R_r| for every r, and
 * r_t = argmax_r u_t(r), ties going to the smallest reference index.  The query stops, without recording, when
 * u_t(r_t) < threshold or when max_matches matches have been recorded.  Otherwise match t - 1 records reference r_t,
 * unique u_t(r_t), intersect |Q_0 n R_{r_t}| and remaining |Q_t| = |Q_{t-1}| - unique, and Q_t = Q_{t-1} \ R_{r_t}.
 * So no reference is picked twice, unique never grows, and the result is a deterministic function of the sketches:
 * a block of queries gives the same rows as the whole call.
 * Outputs: d_n_matches[q] (n_q values, always written: 0 when n_r == 0); match t of query q in slot
 * q * max_matches + t of d_match_ref, d_match_unique, d_match_intersect and d_match_remaining (n_q * max_matches
 * values each); slots past d_n_matches[q] are not written.  Counts are uint32, as in kmerml_fmh_compare.
 * threshold >= 1, max_matches >= 1; n_q == 0 returns at once.
 * Device workspace (the context's, kept between calls): 4 n_q n_r bytes for |Q n R|, then for the n_c candidate
 * references (those with |Q n R| >= threshold for some query) 8 (their total hashes) + 8 n_q n_c bytes, plus
 * 9 (total query hashes) + 24 n_q bytes.  Synchronous: one host read per round.
 */
int kmerml_fmh_gather(kmerml_ctx *ctx, const uint64_t *d_q_hashes, const uint64_t *d_q_offsets, int n_q,
                      const uint64_t *d_r_hashes, const uint64_t *d_r_offsets, int n_r, uint32_t threshold,
                      int max_matches, int32_t *d_n_matches, int32_t *d_match_ref, uint32_t *d_match_unique,
                      uint32_t *d_match_intersect, uint32_t *d_match_remaining, void *stream);
int kmerml_fmh_gather_abundance(kmerml_ctx *ctx, const uint64_t *d_q_hashes, const uint64_t *d_q_offsets, int n_q,
                                const uint64_t *d_r_hashes, const uint64_t *d_r_offsets, int n_r, uint32_t threshold,
                                int max_matches, int32_t *d_n_matches, int32_t *d_match_ref, uint32_t *d_match_unique,
                                uint32_t *d_match_intersect, uint32_t *d_match_remaining,
                                const uint32_t *d_q_abundances, uint64_t *d_match_unique_weighted,
                                uint64_t *d_match_unique_sumsq, double *d_match_median_abund, void *stream);

/*
 * Measurement hooks (bench.py): with profiling enabled every kernel the library
 * launches is bracketed by CUDA events on the launching stream.  kmerml_profile_read
 * synchronises those events and returns the accumulated device time per kernel family
 * and the number of kernel launches since the last reset.
 */
typedef struct kmerml_profile {
    uint64_t launches;        /* all kernels of this library (memsets excluded) */
    uint64_t count_launches;  /* counting-kernel launches */
    double ms_count;          /* device time inside the counting kernels */
    double ms_cascade;        /* ... the marginalisation cascade */
    double ms_finalize;       /* ... fold / normalise */
    double ms_other;          /* prologue and the rest */
    double ms_partition;      /* ... the partition kernel (k = 9..12) */
    double ms_bucket;         /* ... the bucket histogram + in-bucket cascade kernel */
} kmerml_profile;
int kmerml_profile_enable(kmerml_ctx *ctx, int on);
int kmerml_profile_read(kmerml_ctx *ctx, kmerml_profile *out, int reset);

#ifdef __cplusplus
}
#endif
#endif /* KMERML_B200_H */
