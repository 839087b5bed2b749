// internal.h -- declarations shared by the translation units of libkmerml_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <functional>
#include <string>

#include "../../include/kmerml_b200.h"

namespace km {

// ---- error plumbing (thread-local message, never throws across the C-ABI) ----
void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
#define KM_CUDA(expr)                                        \
    do {                                                     \
        cudaError_t e__ = (expr);                            \
        if (e__ != cudaSuccess) return ::km::cuda_fail(e__, #expr); \
    } while (0)

// ---- device-side descriptors --------------------------------------------------
struct GenomeDev {            // one genome's byte range inside the batch buffer
    uint64_t file_lo;         // start of the file
    uint64_t lo;              // first header line (set by the prologue kernel)
    uint64_t hi;              // end of the file
};

struct GenomeStats {          // per genome, zeroed by the prologue kernel
    unsigned long long total_top;     // windows counted at the top (largest) level
    unsigned long long n_tail[16];    // run-end tails per level
};

struct Slice {                // unit of work of one CTA: bytes [begin, end) of one genome
    uint32_t genome;
    uint32_t prev_ok;         // slice_header_kernel: the 32-byte chunk before `begin` is a clean sequence chunk
    uint64_t begin, end;      // multiples of the tile size (absolute buffer offsets)
    uint64_t hdr_until;       // slice_header_kernel: `begin` lies in a header line that ends here (else 0)
    uint32_t prev16;          // ... and these are its last 16 bases (the carry of the slice's first chunk)
    uint64_t line_start;      // slice_header_kernel: start of the line holding `begin` (LS_UNRESOLVED: long line)
    uint64_t scan_last;       // slice_long_scan_kernel: last line start inside the slice before (long lines only)
};

// Where level j (the 4^j histogram) of genome g lives: inside the caller's counts
// row when k=j was requested, else in the context's scratch (cascade pass-through).
struct LevelMap {
    long long off[16];        // >= 0: element offset in the counts row; < 0: -(1 + offset) in scratch
    uint32_t* counts;
    uint64_t counts_stride;
    uint32_t* scratch;
    uint64_t scratch_stride;
    uint32_t scratch_slots;
#ifdef __CUDACC__
    __host__ __device__ __forceinline__ uint32_t* ptr(uint32_t g, int j) const {
        long long o = off[j];
        return o >= 0 ? counts + (uint64_t)g * counts_stride + (uint64_t)o
                      : scratch + (uint64_t)(g % scratch_slots) * scratch_stride + (uint64_t)(-1 - o);
    }
#endif
};

struct RowSpec {              // the caller's k_list, in row order
    int nk;
    int k[16];
    unsigned long long off[17];   // element offset of each k inside a row; off[nk] = row length
};

// ---- launchers (dense.cu) -----------------------------------------------------
constexpr int COUNT_THREADS = 512;                 // threads per CTA of the counting kernels
constexpr int TILE_BYTES = COUNT_THREADS * 32;     // bytes per tile (32-byte chunk per thread)
constexpr int SMEM_MAX_K = 7;                      // 4^7 * 4 B = 64 KB shared histogram

int launch_prologue(const uint8_t* d_fasta, const uint64_t* d_offsets, GenomeDev* d_genomes,
                    GenomeStats* d_stats, int n_genomes, cudaStream_t s);
// d_slices holds n_slices + 1 entries: the last one is scratch (its `genome` field must be 0 on entry).
int launch_slice_headers(const uint8_t* d_fasta, const GenomeDev* d_genomes, Slice* d_slices, int n_slices,
                         cudaStream_t s);
int launch_count(const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices,
                 int n_slices, int k, int k_bottom, int min_rec, bool use_smem, const LevelMap& lm,
                 GenomeStats* d_stats, cudaStream_t s);
int launch_cascade(const LevelMap& lm, int k_top, int k_bottom, uint32_t genome0, int n_genomes,
                   cudaStream_t s);
int cascade_launches(int k_top, int k_bottom);
int finalize_launches(const RowSpec& row, bool canonical);
int launch_finalize(const LevelMap& lm, const RowSpec& row, int k_top, bool canonical,
                    const GenomeStats* d_stats, float* d_freq, uint64_t freq_stride,
                    uint64_t* d_totals, uint32_t genome0, int n_genomes, cudaStream_t s);
// partition path (k = 9..12)
constexpr int PART_MIN_K = 9, PART_MAX_K = 12, PART_LOW_BASES = 7;
constexpr int PART_STAGE_ENTRIES = 32768;               // uint16 payload entries staged per partition CTA (64 KB)
constexpr int PART_MAX_TILES_PER_RUN = 64;              // consecutive tiles one partition CTA walks, at most
uint32_t part_region_cap(int k, int tiles_per_run);     // 32-byte sectors per (run, bucket) region
int launch_partition(const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_runs, int n_runs,
                     int tiles_per_run, int k, int k_bottom, int min_rec, const LevelMap& lm,
                     GenomeStats* d_stats, void* d_payload, uint16_t* d_nsec, uint32_t* d_overflow,
                     unsigned int* d_ov_counts, uint64_t batch_lo, unsigned long long* d_tail_list,
                     unsigned int* d_tail_counts, unsigned int* d_tail_any, uint32_t genome0, cudaStream_t s);
int launch_tails(const uint8_t* d_fasta, const LevelMap& lm, const RowSpec& row, int k, int k_bottom, int min_rec,
                 const GenomeDev* d_genomes, const Slice* d_tiles, int n_tiles, unsigned long long* d_tail_list,
                 unsigned int* d_tail_counts, unsigned int* d_tail_any, uint64_t batch_lo, const GenomeStats* d_stats,
                 float* d_freq, uint64_t freq_stride, uint32_t genome0, int n_genomes, cudaStream_t s);
int launch_bucket(const LevelMap& lm, const RowSpec& row, int k, int k_bottom, const void* d_genome_runs,
                  int tiles_per_run, const void* d_payload, const uint16_t* d_nsec, const GenomeStats* d_stats,
                  float* d_freq, uint64_t freq_stride, uint64_t* d_totals, uint32_t genome0, int n_genomes,
                  cudaStream_t s);
int launch_overflow(const LevelMap& lm, const RowSpec& row, int k, int k_bottom, const GenomeDev* d_genomes,
                    const uint32_t* d_overflow, const unsigned int* d_ov_counts, uint64_t batch_lo,
                    const GenomeStats* d_stats, float* d_freq, uint64_t freq_stride, uint32_t genome0, int n_genomes,
                    cudaStream_t s);
int launch_finalize_low(const LevelMap& lm, const RowSpec& row, int k_top, int level_limit,
                        const GenomeStats* d_stats, float* d_freq, uint64_t freq_stride, uint32_t genome0,
                        int n_genomes, cudaStream_t s);
int launch_encode(const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices, int n_slices,
                  uint8_t* d_symbols, cudaStream_t s);
int launch_first_occurrence(const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices,
                            int n_slices, int k, int min_rec, uint32_t* d_first, cudaStream_t s);
int dense_setup_attributes();

// ---- narrow device -> host wire format (hostpipe.cu) ---------------------------
struct NarrowSpec {           // how a count row maps onto its wire row
    int n, n_small;
    unsigned long long src_off[16];   // narrow levels: element offset inside the count row ...
    unsigned long long dst_off[17];   // ... and byte offset inside the narrow block; dst_off[n] = total
    unsigned char nibble[16];         // 1: two bins per byte (4 bits each, 15 = see the exception list), 0: one byte per bin
    unsigned long long total;         // bytes of the narrow block, a multiple of 16
    unsigned long long small_src[16]; // small levels (uint32 as they are): element offset inside the count row ...
    unsigned long long small_dst[17]; // ... and inside the small block; small_dst[n_small] = small_total
    unsigned long long small_total;
};
int launch_narrow_levels(const uint32_t* d_counts, uint64_t counts_stride, int n_genomes, const NarrowSpec& spec,
                         uint8_t* d_wire, uint64_t wire_stride, uint64_t narrow_off, uint64_t exc_off, uint64_t small_off,
                         uint32_t exc_cap, uint32_t header_magic, uint32_t header_mask, cudaStream_t s);
void widen_u8_to_u32(const uint8_t* src, uint32_t* dst, size_t n);
void widen_u4_to_u32(const uint8_t* src, uint32_t* dst, size_t n_bytes);
class HostPool;
HostPool* host_pool_create(int n_threads);
void host_pool_destroy(HostPool* p);
void host_pool_submit(HostPool* p, std::function<void()> f);
int host_pool_size(const HostPool* p);

// ---- feature CSV text (featcsv.cu) ----------------------------------------------
int launch_parse_kmer_lines(const uint8_t* d_text, const long long* d_line_end, uint64_t n_lines, long long* d_value,
                            long long* d_count, unsigned int* d_bad, cudaStream_t s);
int launch_feature_keys(const long long* d_value, uint64_t n_rows, long long* d_keys, cudaStream_t s);
int launch_feature_line_len(const long long* d_value, const long long* d_count, const long long* d_cls,
                            const int* d_suffix_len, uint64_t n_rows, long long* d_len, cudaStream_t s);
int launch_feature_write(const long long* d_value, const long long* d_count, const long long* d_cls,
                         const long long* d_suffix_off, const int* d_suffix_len, const uint8_t* d_suffix_text,
                         const long long* d_line_off, uint64_t n_rows, uint8_t* d_out, cudaStream_t s);

// ---- reductions (stats.cu) ------------------------------------------------------
size_t count_stats_workspace();
int launch_count_stats(const uint32_t* d_counts, uint64_t n_bins, void* workspace, unsigned long long* d_out, cudaStream_t s);
int launch_column_stats(const void* d_x, int dtype, uint64_t stride, int n_rows, uint64_t m, uint32_t* d_nnz,
                        double* d_mean, double* d_var, cudaStream_t s);

// ---- sparse path (sparse.cu) ---------------------------------------------------
struct SparseWork;
struct SparsePending {        // the reduced result of the last sparse count, still in the workspace (kmerml_sparse_fetch)
    bool valid = false;
    uint64_t* sorted_keys = nullptr;
    uint32_t* sorted_ends = nullptr;
    uint64_t n = 0, nu = 0, cap = 0;
    const void* workspace = nullptr;
};
size_t sparse_workspace_bytes(uint64_t cap);
int sparse_fetch(void* workspace, const SparsePending& p, uint64_t* d_keys_out, uint32_t* d_counts_out,
                 uint32_t* d_first_out, cudaStream_t s);
// The slice table (d_genomes, d_slices, n_slices) covers the whole file in SPARSE_SLICE_BYTES slices; the slices of
// [range_begin, range_end) emit their windows.
int run_sparse_in(void* workspace, const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices, int n_slices,
                  uint64_t range_begin, uint64_t range_end, int k, int min_rec, bool canonical, uint64_t cap,
                  uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap, uint64_t* h_unique,
                  uint64_t* h_windows, SparsePending* pending, cudaStream_t s);
int run_sparse_emit_by_owner(void* workspace, const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices,
                             int n_slices, uint64_t range_begin, uint64_t range_end, int k, int min_rec, bool canonical,
                             int owner_bits, uint64_t cap, uint64_t* d_keys_out, uint32_t* d_ends_out, uint64_t out_cap,
                             uint64_t* h_windows, uint64_t* h_owner_counts, cudaStream_t s);
int run_sparse_reduce_windows(void* workspace, int sort_bits, const uint64_t* d_keys, const uint32_t* d_ends, uint64_t n,
                              uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                              uint64_t* h_unique, SparsePending* pending, cudaStream_t s);

size_t merge_workspace_bytes(uint64_t n);
int run_merge_sparse(void* workspace, int k, const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first,
                     uint64_t n, uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                     uint64_t* h_unique, cudaStream_t s);

// ---- MinHash sketches (sketch.cu) -----------------------------------------------
constexpr uint64_t SPARSE_TILE_BYTES = 8192, SPARSE_SLICE_BYTES = 131072;   // the sparse walker's tile and CTA slice
struct SketchGenome {                 // one genome of a sketch round
    uint64_t tau;                     // windows whose hash is <= tau survive (~0: every window)
    uint64_t region;                  // first slot of the genome's survivor region
    uint64_t cap;                     // slots of that region
    unsigned long long count;         // survivors (zeroed by the host; above cap: the region overflowed)
};
enum : uint32_t { SKETCH_DONE = 0, SKETCH_MORE = 1, SKETCH_OVERFLOW = 2 };    // status of a genome after a round
// the seed term of the hash, added to the key before fmix64
inline uint64_t sketch_seed_add(uint64_t seed) { return 0x9E3779B97F4A7C15ull * (seed + 1); }
int launch_sketch_emit(const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices, int n_slices, int k,
                       int min_rec, bool canonical, uint64_t seed, SketchGenome* d_sg, uint64_t* d_regions, cudaStream_t s);
size_t sketch_sort_temp_bytes(int n_items, int n_segments);
// d_seg: 2 * n_active ints (segment begins | ends), filled here; every active genome's region sorted into d_sorted
int launch_sketch_sort(const SketchGenome* d_sg, const int* d_active, int n_active, int* d_seg, int n_items,
                       const uint64_t* d_regions, uint64_t* d_sorted, void* temp, size_t temp_bytes, cudaStream_t s);
// d_status[i] is the status of genome d_active[i]
int launch_sketch_select(const SketchGenome* d_sg, const int* d_active, int n_active, const uint64_t* d_sorted,
                         int sketch_size, uint64_t* d_sketches, uint64_t stride, uint32_t* d_filled, uint32_t* d_status,
                         cudaStream_t s);
int launch_sketch_distance(const uint64_t* d_sketches, uint64_t stride, const uint32_t* d_filled, int n, int sketch_size,
                           int k, int row_begin, int row_end, int metric, float* d_out32, double* d_out64, cudaStream_t s);
// scaled sketches: per active genome of a sorted round, its survivors (above its region's cap: overflow), the rank of
// its first distinct value among the round's kept values and how many it keeps
struct FmhRoundGenome {
    unsigned long long count, first, distinct;
};
size_t fmh_scan_temp_bytes(int n_items);
// d_flags, d_pos: n_items words each; d_seg as launch_sketch_sort left it
int launch_fmh_distinct(const SketchGenome* d_sg, const int* d_active, int n_active, const int* d_seg, int n_items,
                        const uint64_t* d_sorted, uint32_t* d_flags, uint32_t* d_pos, void* temp, size_t temp_bytes,
                        FmhRoundGenome* d_out, cudaStream_t s);
int launch_fmh_scatter(const uint64_t* d_sorted, const uint32_t* d_flags, const uint32_t* d_pos, int n_items, uint64_t* d_out,
                       cudaStream_t s);
// the run length of every kept slot of a round (KMERML_FLAG_FMH_ABUNDANCE), at d_out[d_pos[slot]] like the scatter
int launch_fmh_abundance(const uint32_t* d_flags, const uint32_t* d_pos, const int* d_seg, int n_active, int n_items,
                         uint32_t* d_out, cudaStream_t s);
// T = uint64_t (values) or uint32_t (abundances)
template <typename T>
int launch_fmh_gather(const T* d_kept, const uint64_t* d_begin, const uint64_t* d_offsets, int n, uint64_t total, T* d_out,
                      cudaStream_t s);
size_t fmh_compare_workspace(int n_r);
int launch_fmh_compare(const uint64_t* d_qh, const uint64_t* d_q_off, int n_q, const uint64_t* d_rh, const uint64_t* d_r_off,
                       int n_r, int k, int metric, int sm_count, void* workspace, uint32_t* d_inter, float* d_out32,
                       double* d_out64, cudaStream_t s);
// weighted metrics: d_num (n_q x n_r) = sum_{Q n R} a_Q (weighted containment) or a_Q a_R (angular similarity)
size_t fmh_compare_weighted_workspace(int n_q, int n_r);
int launch_fmh_compare_weighted(const uint64_t* d_qh, const uint64_t* d_q_off, const uint32_t* d_qa, int n_q,
                                const uint64_t* d_rh, const uint64_t* d_r_off, const uint32_t* d_ra, int n_r, int metric,
                                int sm_count, void* workspace, unsigned long long* d_num, float* d_out32, double* d_out64,
                                cudaStream_t s);
// gather: the candidate flags of a prefetched n_q x n_r intersection matrix (zeroed here) ...
int launch_fmh_greedy_flag(const uint32_t* d_x, int n_q, int n_r, uint32_t threshold, uint8_t* d_flags, cudaStream_t s);
// ... one round's pick of every running query (d_d: the last round's subtraction, unused in round 0) ...
int launch_fmh_greedy_select(uint32_t* d_u, const uint32_t* d_d, int n_c, const uint32_t* d_x, int n_q, int n_r,
                             const int* d_cand, const uint64_t* d_q_off, int round, uint32_t threshold, int max_matches,
                             int* d_pick, uint32_t* d_remaining, unsigned long long* d_s_len, int32_t* d_n_matches,
                             int32_t* d_ref, uint32_t* d_unique, uint32_t* d_inter, uint32_t* d_rem,
                             unsigned int* d_n_picked, cudaStream_t s);
// ... and the hashes each pick takes, as a sorted CSR (d_s_len, d_s_off: n_q + 1 words; d_s_len[n_q] = 0); with `ab`,
// also their query abundances beside them (ab->s_abund) and the sum and sum of squares of those per recorded match
struct GatherAbund {
    const uint32_t* qa;               // query abundances, parallel to the query hashes
    uint32_t* s_abund;                // S_t's abundances, parallel to S_t
    unsigned long long* sum;          // per match slot q * max_matches + round
    unsigned long long* sumsq;
    int round, max_matches;
};
size_t fmh_greedy_scan_temp_bytes(int n_q);
int launch_fmh_greedy_remove(const uint64_t* d_qh, const uint64_t* d_q_off, int n_q, const uint64_t* d_ch,
                             const uint64_t* d_c_off, const int* d_pick, const unsigned long long* d_s_len,
                             unsigned long long* d_s_off, void* temp, size_t temp_bytes, uint8_t* d_assigned,
                             uint64_t* d_s_hashes, unsigned int* d_bad, const GatherAbund* ab, cudaStream_t s);
// ... and the median of S_t's abundances of every query that recorded a match this round (total = |S_t| summed)
size_t fmh_greedy_median_temp_bytes(int n_q, int total);
int launch_fmh_greedy_median(const GatherAbund& ab, const unsigned long long* d_s_off, const int* d_pick, int n_q,
                             int total, uint32_t* d_sorted, void* temp, size_t temp_bytes, double* d_median,
                             cudaStream_t s);

// ---- k{k}.txt text (format.cu) --------------------------------------------------
size_t format_workspace_bytes(uint64_t n_bins, uint64_t max_lines);
int run_format_dense(void* workspace, int k, const uint32_t* d_counts, const uint32_t* d_first, bool canonical,
                     uint64_t max_lines, uint8_t* d_text, uint64_t text_cap, uint64_t* h_len, uint64_t* h_lines,
                     cudaStream_t s);
int run_format_lines(void* workspace, int k, const uint64_t* d_codes, const uint32_t* d_counts, uint64_t n,
                     uint8_t* d_text, uint64_t text_cap, uint64_t* h_len, cudaStream_t s);

// ---- launchers (features.cu) --------------------------------------------------
int launch_scan_records(const uint8_t* d_fasta, uint64_t nbytes, int need, unsigned long long* d_offsets,
                        uint8_t* d_short, uint32_t cap, uint32_t* d_count, cudaStream_t s);
int launch_record_short(const uint8_t* d_fasta, uint64_t nbytes, const unsigned long long* d_offsets, uint32_t n,
                        int need, uint8_t* d_short, cudaStream_t s);
int launch_genome_stats(const uint8_t* d_fasta, uint64_t nbytes, unsigned long long* d_out, cudaStream_t s);
int launch_static_features(int k, int compat, int32_t* d_out, cudaStream_t s);
int launch_normalize_rows(const uint32_t* d_counts, uint64_t counts_stride, const uint64_t* d_totals, int n_rows,
                          uint64_t m, float* d_out, uint64_t out_stride, cudaStream_t s);
int launch_pairwise(const void* d_x, int dtype, uint64_t stride, int n, uint64_t m, int metric, double* d_gram,
                    float* d_out32, double* d_out64, cudaStream_t s);

// ---- distances of count rows from the exact tensor-core Gram (gram_tc.cu) ---------
int launch_count_planes(const uint32_t* d_counts, uint64_t stride, int n, uint64_t m, uint8_t* d_planes,
                        uint64_t plane_stride, double* d_sumsq, unsigned int* d_max, cudaStream_t s);
size_t distance_rows_workspace(int n, uint64_t m);
int launch_distance_rows_planes(const uint8_t* d_planes, uint64_t plane_stride, int n_planes, int n, uint64_t m,
                                const double* d_sumsq, int row_begin, int row_end, int metric, void* workspace,
                                float* d_out32, double* d_out64, cudaStream_t s);
int launch_distance_rows_tc(const uint32_t* d_counts, uint64_t stride, int n, uint64_t m, int row_begin, int row_end,
                            int metric, void* workspace, float* d_out32, double* d_out64, cudaStream_t s);

#ifdef __CUDACC__
// Distance of rows i != j from their Gram entries -- metric 0: cosine 1 - G_ij / sqrt(G_ii G_jj) (NaN when a row is
// all zero); 1: Euclidean sqrt(G_ii + G_jj - 2 G_ij).  The one formula of distance_rows_kernel (exact Gram of count
// rows) and distance_from_gram_kernel (fp64 Gram).
__device__ __forceinline__ double gram_distance(double gii, double gjj, double gij, int metric) {
    if (metric == 0) {
        const double den = sqrt(gii) * sqrt(gjj);
        return den > 0.0 ? 1.0 - gij / den : nan("");
    }
    const double d2 = gii + gjj - 2.0 * gij;
    return d2 > 0.0 ? sqrt(d2) : 0.0;
}
#endif

}  // namespace km
