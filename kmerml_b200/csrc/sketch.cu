// sketch.cu -- bottom-s MinHash sketches of whole genomes for any k <= 32, and the Mash / Jaccard distances of
// those sketches (Ondov et al. 2016).  The hash is h(key) = fmix64(key + 0x9E3779B97F4A7C15 (seed + 1)) of the 2-bit
// packed (canonical) k-mer; it is a bijection, so distinct hashes are distinct k-mers.  The sketches are this
// library's own: not file-compatible with Mash or sourmash.
//
//   sketch_emit_kernel      the sparse path's walker (sparse_walk.cuh) over a multi-genome slice table; a window is
//                           kept when its hash is <= the genome's threshold tau, appended to the genome's own region
//                           with one warp-aggregated reservation.  tau is chosen so that ~3 s windows survive.
//   CUB segmented sort      every genome's survivors, ascending
//   sketch_select_kernel    the first s distinct values of each genome, its fill count and a status: done, too few
//                           distinct survivors below tau (run again with a larger tau), or region overflow (run again
//                           with a region of one slot per byte).  The host loop is kmerml_sketch_batch (api.cu).
//   sketch_distance_kernel  rows [row_begin, row_end) x all n columns of the distance matrix, exact and symmetric.
//
// Scaled (FracMinHash) sketches (Irber et al. 2022) keep every distinct hash <= T = (2^64 - 1) / scale, so their size
// grows with the genome and one genome's containment in another can be estimated.  They reuse the emitter and the
// segmented sort with tau = T for every genome (the same host round loop, sketch_rounds in api.cu), then
//   fmh_flag_kernel + CUB scan + fmh_round_kernel   which sorted slots are distinct values, and where each genome's
//                           values go among the round's kept values; a region overflow runs again with exactly the
//                           survivors the cursor counted
//   fmh_scatter_kernel      the kept values of a round, appended to a buffer of the context
//   fmh_gather_kernel       that buffer in genome order, as CSR
//   fmh_intersect_kernel    exact |Q n R| of every (query, reference) pair of two sets of scaled sketches, and
//   fmh_metric_kernel       containment, max-containment, Jaccard or containment ANI (Hera et al. 2023) from it.
// Gather (Irber et al. 2022) splits each query greedily into the references that cover it, in rounds over all queries:
//   fmh_greedy_flag_kernel    the candidate references, from a prefetched |Q n R| (fmh_intersect_kernel)
//   fmh_greedy_select_kernel  per query, the candidate with the most still-unassigned hashes (ties: smallest index)
//   fmh_greedy_remove_kernel  per query, the hashes that pick takes: marked assigned and listed as a sorted CSR, which
//                             fmh_intersect_kernel then subtracts from every candidate's count.
// Abundances (KMERML_FLAG_FMH_ABUNDANCE): fmh_abundance_kernel writes each kept value's run length in the sorted round
// beside it; fmh_intersect_kernel<true> + fmh_abund_sums_kernel + fmh_weighted_metric_kernel give weighted containment
// and angular similarity; fmh_greedy_remove_kernel<true> sums S_t's query abundances, and a CUB segmented sort +
// fmh_greedy_median_kernel give their median.
#include <cub/cub.cuh>

#include "sparse_walk.cuh"

namespace km {

__host__ __device__ __forceinline__ uint64_t fmix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}

// Survivors of one genome: hashes <= tau go to its region; the cursor counts every survivor, so a count above the
// region's capacity reports the overflow.
struct SketchSink {
    uint64_t* region;
    unsigned long long* cursor;
    uint64_t cap, tau, seed_add;
    struct Lanes {};
    __device__ __forceinline__ Lanes fast_begin(bool, unsigned, unsigned, int) const { return Lanes{}; }
    __device__ __forceinline__ void fast_window(const Lanes&, int, uint64_t key, uint64_t pos) const { window(key, pos); }
    __device__ __forceinline__ void window(uint64_t key, uint64_t) const {
        const uint64_t h = fmix64(key + seed_add);
        if (h > tau) return;
        const unsigned active = __activemask();
        const int lane = threadIdx.x & 31;
        const int leader = __ffs(active) - 1;
        unsigned long long b = 0;
        if (lane == leader) b = atomicAdd(cursor, (unsigned long long)__popc(active));
        b = __shfl_sync(active, b, leader);
        const unsigned long long slot = b + __popc(active & ((1u << lane) - 1u));
        if (slot < cap) region[slot] = h;
    }
};

__global__ void __launch_bounds__(SPARSE_THREADS)
sketch_emit_kernel(const uint8_t* __restrict__ buf, const GenomeDev* __restrict__ gds, const Slice* __restrict__ slices,
                   SparseParams P, uint64_t seed_add, SketchGenome* sg, uint64_t* regions) {
    const Slice sl = slices[blockIdx.x];
    const GenomeDev gd = gds[sl.genome];
    SketchGenome* me = sg + sl.genome;
    SketchSink sink;
    sink.region = regions + me->region;
    sink.cursor = &me->count;
    sink.cap = me->cap;
    sink.tau = me->tau;
    sink.seed_add = seed_add;
    walk_sparse_slice(buf, gd, sl, P, sink);
}

// Segment i of the sort = the filled part of the region of genome active[i].
__global__ void sketch_segments_kernel(const SketchGenome* __restrict__ sg, const int* __restrict__ active, int n_active,
                                       int* seg_begin, int* seg_end) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_active) return;
    const SketchGenome me = sg[active[i]];
    seg_begin[i] = (int)me.region;
    seg_end[i] = (int)(me.region + (me.count < me.cap ? me.count : me.cap));
}

constexpr int SELECT_THREADS = 256;

__global__ void __launch_bounds__(SELECT_THREADS)
sketch_select_kernel(const uint64_t* __restrict__ sorted, const SketchGenome* __restrict__ sg, const int* __restrict__ active,
                     int s, uint64_t* sketches, uint64_t stride, uint32_t* filled, uint32_t* status) {
    using Scan = cub::BlockScan<int, SELECT_THREADS>;
    __shared__ typename Scan::TempStorage tmp;
    const int tid = threadIdx.x;
    const int g = active[blockIdx.x];
    const SketchGenome me = sg[g];
    if (me.count > me.cap) {
        if (tid == 0) status[blockIdx.x] = SKETCH_OVERFLOW;
        return;
    }
    const uint64_t* v = sorted + me.region;
    uint64_t* out = sketches + (uint64_t)g * stride;
    int kept = 0;                                     // distinct values so far (the same in every thread)
    for (uint64_t base = 0; base < me.count && kept < s; base += SELECT_THREADS) {
        const uint64_t i = base + tid;
        const int first = (i < me.count && (i == 0 || v[i] != v[i - 1])) ? 1 : 0;
        int rank, total;
        Scan(tmp).ExclusiveSum(first, rank, total);
        if (first && kept + rank < s) out[kept + rank] = v[i];
        kept += total;
        __syncthreads();
    }
    const int f = kept < s ? kept : s;
    for (int i = f + tid; i < s; i += SELECT_THREADS) out[i] = ~0ull;
    if (tid == 0) {
        filled[g] = (uint32_t)f;
        status[blockIdx.x] = (kept < s && me.tau != ~0ull) ? SKETCH_MORE : SKETCH_DONE;
    }
}

int launch_sketch_emit(const uint8_t* d_fasta, const GenomeDev* d_genomes, const Slice* d_slices, int n_slices, int k,
                       int min_rec, bool canonical, uint64_t seed, SketchGenome* d_sg, uint64_t* d_regions, cudaStream_t s) {
    if (n_slices <= 0) return KMERML_OK;
    SparseParams P;
    P.k = k;
    P.min_rec = min_rec;
    P.canonical = canonical ? 1 : 0;
    P.mask = k >= 32 ? ~0ull : ((1ull << (2 * k)) - 1ull);
    sketch_emit_kernel<<<n_slices, SPARSE_THREADS, 0, s>>>(d_fasta, d_genomes, d_slices, P, sketch_seed_add(seed), d_sg,
                                                           d_regions);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

size_t sketch_sort_temp_bytes(int n_items, int n_segments) {
    size_t t = 0;
    cub::DeviceSegmentedSort::SortKeys(nullptr, t, (const uint64_t*)nullptr, (uint64_t*)nullptr, n_items, n_segments,
                                       (const int*)nullptr, (const int*)nullptr);
    return t;
}

int launch_sketch_sort(const SketchGenome* d_sg, const int* d_active, int n_active, int* d_seg, int n_items,
                       const uint64_t* d_regions, uint64_t* d_sorted, void* temp, size_t temp_bytes, cudaStream_t s) {
    if (n_active <= 0) return KMERML_OK;
    int* seg_begin = d_seg;
    int* seg_end = d_seg + n_active;
    sketch_segments_kernel<<<(n_active + 255) / 256, 256, 0, s>>>(d_sg, d_active, n_active, seg_begin, seg_end);
    KM_CUDA(cudaGetLastError());
    size_t tb = temp_bytes;
    KM_CUDA(cub::DeviceSegmentedSort::SortKeys(temp, tb, d_regions, d_sorted, n_items, n_active, (const int*)seg_begin,
                                               (const int*)seg_end, s));
    return KMERML_OK;
}

int launch_sketch_select(const SketchGenome* d_sg, const int* d_active, int n_active, const uint64_t* d_sorted,
                         int sketch_size, uint64_t* d_sketches, uint64_t stride, uint32_t* d_filled, uint32_t* d_status,
                         cudaStream_t s) {
    if (n_active <= 0) return KMERML_OK;
    sketch_select_kernel<<<n_active, SELECT_THREADS, 0, s>>>(d_sorted, d_sg, d_active, sketch_size, d_sketches, stride,
                                                             d_filled, d_status);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

// ---- distances ---------------------------------------------------------------------------------------------------
// D from x = |U n A n B| and |U| (U = the min(s, |A u B|) smallest values of A u B); j = x / |U|.
__device__ __forceinline__ double sketch_metric(int x, int u, int k, int metric) {
    if (x == 0) return 1.0;                           // j = 0, also |U| = 0 (two empty sketches)
    if (x == u) return 0.0;                           // j = 1
    const double j = (double)x / (double)u;
    return metric == KMERML_SKETCH_METRIC_JACCARD ? 1.0 - j : -log(2.0 * j / (1.0 + j)) / (double)k;
}

constexpr int SKD_THREADS = 256;
constexpr int SKD_ROWS = 64;                          // rows one CTA compares with its column

// One CTA per (column j, block of SKD_ROWS rows): the sketch B of column j sits in shared memory, one warp per row i
// walks A = sketch i 32 values at a time.  For a_t in A, r_t = |{b in B : b < a_t}| (binary search) and c_t = the
// number of earlier a found in B (a ballot prefix): a_t is the (t + r_t - c_t)-th smallest value of A u B, so it is
// in U iff that rank is < s, and it counts towards x iff it is also found in B.  Ranks grow along A, so the walk
// stops at the first rank >= s (|U| = s then); otherwise |U| = min(s, |A| + |B| - shared).  x and |U| are exact
// integers that do not depend on which sketch is the row: D(i, j) == D(j, i) bit for bit, and a row block is the
// same rows of the whole matrix.
__global__ void __launch_bounds__(SKD_THREADS)
sketch_distance_kernel(const uint64_t* __restrict__ sk, uint64_t stride, const uint32_t* __restrict__ filled, int n, int s,
                       int k, int row_begin, int row_end, int metric, float* out32, double* out64) {
    extern __shared__ uint64_t s_b[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int col = blockIdx.x;
    const int nb = (int)min(filled[col], (uint32_t)s);
    const uint64_t* B = sk + (uint64_t)col * stride;
    for (int t = tid; t < nb; t += SKD_THREADS) s_b[t] = B[t];
    __syncthreads();
    const int r_lo = row_begin + blockIdx.y * SKD_ROWS;
    const int r_hi = min(r_lo + SKD_ROWS, row_end);
    const unsigned below = (1u << lane) - 1u;
    for (int row = r_lo + warp; row < r_hi; row += SKD_THREADS / 32) {
        const int na = (int)min(filled[row], (uint32_t)s);
        const uint64_t* A = sk + (uint64_t)row * stride;
        int shared = 0, x = 0;
        bool full = false;
        for (int a0 = 0; a0 < na; a0 += 32) {
            const int t = a0 + lane;
            const bool valid = t < na;
            const uint64_t a = valid ? A[t] : 0;
            int lo = 0, hi = nb;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (s_b[mid] < a) lo = mid + 1; else hi = mid;
            }
            const bool found = valid && lo < nb && s_b[lo] == a;
            const unsigned fm = __ballot_sync(0xffffffffu, found);
            const int rank = t + lo - (shared + __popc(fm & below));
            x += __popc(__ballot_sync(0xffffffffu, found && rank < s));
            shared += __popc(fm);
            if (__any_sync(0xffffffffu, valid && rank >= s)) { full = true; break; }
        }
        if (lane == 0) {
            const int u = full ? s : min(s, na + nb - shared);
            const double d = sketch_metric(x, u, k, metric);
            const uint64_t o = (uint64_t)(row - row_begin) * n + col;
            if (out64) out64[o] = d;
            if (out32) out32[o] = (float)d;
        }
    }
}

int launch_sketch_distance(const uint64_t* d_sketches, uint64_t stride, const uint32_t* d_filled, int n, int sketch_size,
                           int k, int row_begin, int row_end, int metric, float* d_out32, double* d_out64, cudaStream_t s) {
    if (row_begin >= row_end || n <= 0) return KMERML_OK;
    const size_t smem = (size_t)sketch_size * 8;
    KM_CUDA(cudaFuncSetAttribute(sketch_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((unsigned)n, (unsigned)((row_end - row_begin + SKD_ROWS - 1) / SKD_ROWS));
    if (grid.y > 65535) {
        set_error("sketch distance: more than 65535 x 64 rows in one call");
        return KMERML_ERR_RANGE;
    }
    sketch_distance_kernel<<<grid, SKD_THREADS, smem, s>>>(d_sketches, stride, d_filled, n, sketch_size, k, row_begin,
                                                           row_end, metric, d_out32, d_out64);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

// ---- scaled (FracMinHash) sketches ------------------------------------------------------------------------------
// A sorted round keeps slot i when it is a distinct value of a genome whose region did not overflow: the first slot of
// the genome's segment, or one that differs from the slot before it.  The genome of slot i is the last active genome
// whose segment begins at or before i (segments ascend with the active index; empty ones included).
__global__ void fmh_flag_kernel(const uint64_t* __restrict__ sorted, const SketchGenome* __restrict__ sg,
                                const int* __restrict__ active, const int* __restrict__ seg_begin,
                                const int* __restrict__ seg_end, int n_active, int n_items, uint32_t* flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    int lo = 0, hi = n_active;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (seg_begin[mid] <= i) lo = mid + 1; else hi = mid;
    }
    const int j = lo - 1;                             // >= 0: the first segment begins at slot 0
    const SketchGenome me = sg[active[j]];
    flags[i] = (i < seg_end[j] && me.count <= me.cap && (i == seg_begin[j] || sorted[i] != sorted[i - 1])) ? 1u : 0u;
}

// Per active genome: its survivors, the rank of its first distinct value among the round's kept values, and how many
// it keeps (0 after an overflow).
__global__ void fmh_round_kernel(const SketchGenome* __restrict__ sg, const int* __restrict__ active,
                                 const int* __restrict__ seg_begin, const int* __restrict__ seg_end, int n_active,
                                 const uint32_t* __restrict__ flags, const uint32_t* __restrict__ pos, FmhRoundGenome* out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_active) return;
    const int b = seg_begin[j], e = seg_end[j];
    FmhRoundGenome r;
    r.count = sg[active[j]].count;
    r.first = e > b ? pos[b] : 0;
    r.distinct = e > b ? (unsigned long long)pos[e - 1] + flags[e - 1] - pos[b] : 0;
    out[j] = r;
}

__global__ void fmh_scatter_kernel(const uint64_t* __restrict__ sorted, const uint32_t* __restrict__ flags,
                                   const uint32_t* __restrict__ pos, int n_items, uint64_t* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_items && flags[i]) out[pos[i]] = sorted[i];
}

// Abundance of kept slot i (KMERML_FLAG_FMH_ABUNDANCE): the length of its run of equal sorted survivors, i.e. the next
// kept slot of its segment (or the segment end) minus i, written beside the value fmh_scatter_kernel writes.  Kept slots
// after i carry pos + flag > pos[i] + 1, so the run end is a binary search over the inclusive scan pos + flags.
__global__ void fmh_abundance_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ pos,
                                     const int* __restrict__ seg_begin, const int* __restrict__ seg_end, int n_active,
                                     int n_items, uint32_t* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items || !flags[i]) return;
    int lo = 0, hi = n_active;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (seg_begin[mid] <= i) lo = mid + 1; else hi = mid;
    }
    const int end = seg_end[lo - 1];
    const uint32_t next = pos[i] + 1;
    int a = i + 1, b = end;                           // the first slot in [i + 1, end) that is kept, else end
    while (a < b) {
        const int mid = (a + b) >> 1;
        if (pos[mid] + flags[mid] > next) b = mid; else a = mid + 1;
    }
    out[pos[i]] = (uint32_t)(a - i);
}

// out[offsets[g] + t] = kept[begin[g] + t] for t < offsets[g + 1] - offsets[g]: the kept values (or their abundances)
// in genome order.
template <typename T>
__global__ void fmh_gather_kernel(const T* __restrict__ kept, const uint64_t* __restrict__ begin,
                                  const uint64_t* __restrict__ offsets, int n, uint64_t total, T* out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        int lo = 0, hi = n;                           // the last genome whose output begins at or before i
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (offsets[mid] <= i) lo = mid + 1; else hi = mid;
        }
        const int g = lo - 1;
        out[i] = kept[begin[g] + (i - offsets[g])];
    }
}

size_t fmh_scan_temp_bytes(int n_items) {
    size_t t = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, t, (const uint32_t*)nullptr, (uint32_t*)nullptr, n_items);
    return t;
}

int launch_fmh_distinct(const SketchGenome* d_sg, const int* d_active, int n_active, const int* d_seg, int n_items,
                        const uint64_t* d_sorted, uint32_t* d_flags, uint32_t* d_pos, void* temp, size_t temp_bytes,
                        FmhRoundGenome* d_out, cudaStream_t s) {
    if (n_active <= 0) return KMERML_OK;
    if (n_items > 0) {
        fmh_flag_kernel<<<(n_items + 255) / 256, 256, 0, s>>>(d_sorted, d_sg, d_active, d_seg, d_seg + n_active, n_active,
                                                             n_items, d_flags);
        KM_CUDA(cudaGetLastError());
        size_t tb = temp_bytes;
        KM_CUDA(cub::DeviceScan::ExclusiveSum(temp, tb, d_flags, d_pos, n_items, s));
    }
    fmh_round_kernel<<<(n_active + 255) / 256, 256, 0, s>>>(d_sg, d_active, d_seg, d_seg + n_active, n_active, d_flags,
                                                            d_pos, d_out);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

int launch_fmh_scatter(const uint64_t* d_sorted, const uint32_t* d_flags, const uint32_t* d_pos, int n_items, uint64_t* d_out,
                       cudaStream_t s) {
    if (n_items <= 0) return KMERML_OK;
    fmh_scatter_kernel<<<(n_items + 255) / 256, 256, 0, s>>>(d_sorted, d_flags, d_pos, n_items, d_out);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

int launch_fmh_abundance(const uint32_t* d_flags, const uint32_t* d_pos, const int* d_seg, int n_active, int n_items,
                         uint32_t* d_out, cudaStream_t s) {
    if (n_items <= 0) return KMERML_OK;
    fmh_abundance_kernel<<<(n_items + 255) / 256, 256, 0, s>>>(d_flags, d_pos, d_seg, d_seg + n_active, n_active, n_items,
                                                               d_out);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

template <typename T>
int launch_fmh_gather(const T* d_kept, const uint64_t* d_begin, const uint64_t* d_offsets, int n, uint64_t total, T* d_out,
                      cudaStream_t s) {
    if (!total) return KMERML_OK;
    const uint64_t blocks = std::min<uint64_t>((total + 255) / 256, 1ull << 16);
    fmh_gather_kernel<T><<<(unsigned)blocks, 256, 0, s>>>(d_kept, d_begin, d_offsets, n, total, d_out);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}
template int launch_fmh_gather<uint64_t>(const uint64_t*, const uint64_t*, const uint64_t*, int, uint64_t, uint64_t*,
                                         cudaStream_t);
template int launch_fmh_gather<uint32_t>(const uint32_t*, const uint64_t*, const uint64_t*, int, uint64_t, uint32_t*,
                                         cudaStream_t);

// ---- |Q n R| of two sets of scaled sketches ----------------------------------------------------------------------
constexpr int FMH_THREADS = 256;
constexpr int FMH_CHUNK = 8192;                       // reference values one CTA holds in shared memory (64 KB)
constexpr int FMH_QROWS = 32;                         // queries one CTA compares with its chunk
constexpr int FMH_BUCKET_BITS = 11;                   // 2048 buckets index the chunk (8 KB)
constexpr size_t FMH_SMEM = (size_t)FMH_CHUNK * 8 + ((1u << FMH_BUCKET_BITS) + 1) * 4;

// chunks[r] = ceil(|R_r| / FMH_CHUNK), prefix[r] = chunks before reference r, prefix[n_r] = all chunks (one CTA).
__global__ void __launch_bounds__(SELECT_THREADS)
fmh_chunk_prefix_kernel(const uint64_t* __restrict__ r_off, int n_r, unsigned long long* prefix) {
    using Scan = cub::BlockScan<unsigned long long, SELECT_THREADS>;
    __shared__ typename Scan::TempStorage tmp;
    unsigned long long carry = 0;
    for (int base = 0; base < n_r; base += SELECT_THREADS) {
        const int r = base + threadIdx.x;
        const unsigned long long c = r < n_r ? (r_off[r + 1] - r_off[r] + FMH_CHUNK - 1) / FMH_CHUNK : 0;
        unsigned long long x, total;
        Scan(tmp).ExclusiveSum(c, x, total);
        if (r < n_r) prefix[r] = carry + x;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) prefix[n_r] = carry;
}

// First index in [lo, hi) of the ascending list A whose value is >= x (hi if none), the same in every lane: 32 probes
// per step cut the range into 33 parts, so a list of millions takes four or five dependent loads.
__device__ __forceinline__ uint64_t warp_lower_bound(const uint64_t* __restrict__ A, uint64_t lo, uint64_t hi, uint64_t x,
                                                     int lane) {
    while (hi - lo > 32) {
        const uint64_t p = lo + (hi - lo) * (uint64_t)(lane + 1) / 33;
        const int c = __popc(__ballot_sync(0xffffffffu, A[p] < x));
        const uint64_t below = __shfl_sync(0xffffffffu, p, c ? c - 1 : 0);
        const uint64_t above = __shfl_sync(0xffffffffu, p, c < 32 ? c : 31);
        if (c) lo = below + 1;
        if (c < 32) hi = above;
    }
    const uint64_t p = lo + lane;
    return lo + __popc(__ballot_sync(0xffffffffu, p < hi && A[p] < x));
}

// Work item = (chunk of FMH_CHUNK values of one reference, block of FMH_QROWS queries); CTAs stride over the items, so
// a long reference is spread over many CTAs and the query count is not bounded by the grid.  The chunk sits in shared
// memory with an index of 2^FMH_BUCKET_BITS buckets of (value - chunk min) >> shift; a warp per query finds the part
// of its sketch inside [chunk min, chunk max] with two warp-wide searches in global memory, then looks up 32 values at
// a time (index, then a binary search inside the bucket) and counts the hits with a ballot.  The chunks of a reference
// split its values, so their partial counts add up to |Q n R| exactly (one atomic per query and chunk).
// WEIGHTED: a hit adds a_Q (ra NULL) or a_Q a_R instead of 1, in uint64 (the sums fit: see kmerml_fmh_compare_weighted);
// a_R is read from global memory at the hit's chunk position.  Three CTAs share an SM (shared memory), which lets the
// weighted instantiation keep its 64-bit sums in registers; the unweighted one keeps the register choice it had.
template <bool WEIGHTED>
__global__ void __launch_bounds__(FMH_THREADS, WEIGHTED ? 3 : 0)
fmh_intersect_kernel(const uint64_t* __restrict__ qh, const uint64_t* __restrict__ q_off, int n_q,
                     const uint64_t* __restrict__ rh, const uint64_t* __restrict__ r_off, int n_r,
                     const unsigned long long* __restrict__ prefix,
                     std::conditional_t<WEIGHTED, unsigned long long, uint32_t>* inter,
                     const uint32_t* __restrict__ qa, const uint32_t* __restrict__ ra) {
    extern __shared__ uint64_t s_r[];
    uint32_t* s_idx = (uint32_t*)(s_r + FMH_CHUNK);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long n_qb = (unsigned long long)(n_q + FMH_QROWS - 1) / FMH_QROWS;
    const unsigned long long n_items = prefix[n_r] * n_qb;
    for (unsigned long long item = blockIdx.x; item < n_items; item += gridDim.x) {
        const unsigned long long c = item / n_qb;
        const int qb = (int)(item % n_qb);
        int lo = 0, hi = n_r - 1;                     // the reference of chunk c: the last one whose chunks begin <= c
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (prefix[mid] <= c) lo = mid; else hi = mid - 1;
        }
        const int r = lo;
        const uint64_t c_lo = r_off[r] + (c - prefix[r]) * FMH_CHUNK;
        const int len = (int)min((uint64_t)FMH_CHUNK, r_off[r + 1] - c_lo);
        __syncthreads();                              // the previous item is done with the chunk
        for (int t = tid; t < len; t += FMH_THREADS) s_r[t] = rh[c_lo + t];
        __syncthreads();
        const uint64_t cmin = s_r[0], cmax = s_r[len - 1];
        const uint64_t span = cmax - cmin;
        const int bits = span ? 64 - __clzll((long long)span) : 0;
        const int shift = bits > FMH_BUCKET_BITS ? bits - FMH_BUCKET_BITS : 0;
        for (int t = tid; t < len; t += FMH_THREADS) {      // s_idx[b] = first position of bucket >= b
            const int b = (int)((s_r[t] - cmin) >> shift);
            const int bp = t ? (int)((s_r[t - 1] - cmin) >> shift) : -1;
            for (int bb = bp + 1; bb <= b; bb++) s_idx[bb] = t;
            if (t == len - 1) s_idx[b + 1] = len;
        }
        __syncthreads();
        const int q_end = min(n_q, (qb + 1) * FMH_QROWS);
        for (int q = qb * FMH_QROWS + warp; q < q_end; q += FMH_THREADS / 32) {
            const uint64_t* Q = qh + q_off[q];
            const uint64_t nq = q_off[q + 1] - q_off[q];
            const uint64_t a = warp_lower_bound(Q, 0, nq, cmin, lane);
            const uint64_t e = cmax == ~0ull ? nq : warp_lower_bound(Q, a, nq, cmax + 1, lane);
            uint32_t hits = 0;
            unsigned long long mass = 0;              // WEIGHTED: this lane's share of the weighted count
            for (uint64_t t0 = a; t0 < e; t0 += 32) {
                const uint64_t t = t0 + lane;
                bool found = false;
                if (t < e) {
                    const uint64_t v = Q[t];
                    const int b = (int)((v - cmin) >> shift);
                    int l = (int)s_idx[b], h = (int)s_idx[b + 1];
                    const int h0 = h;
                    while (l < h) {
                        const int mid = (l + h) >> 1;
                        if (s_r[mid] < v) l = mid + 1; else h = mid;
                    }
                    found = l < h0 && s_r[l] == v;
                    if constexpr (WEIGHTED) {
                        if (found) mass += (unsigned long long)qa[q_off[q] + t] * (ra ? ra[c_lo + l] : 1u);
                    }
                }
                if constexpr (!WEIGHTED) hits += __popc(__ballot_sync(0xffffffffu, found));
            }
            if constexpr (WEIGHTED) {
                for (int o = 16; o; o >>= 1) mass += __shfl_xor_sync(0xffffffffu, mass, o);
                if (lane == 0 && mass) atomicAdd(inter + (uint64_t)q * n_r + r, mass);
            } else {
                if (lane == 0 && hits) atomicAdd(inter + (uint64_t)q * n_r + r, hits);
            }
        }
    }
}

// The metric of x = |Q n R| (float64; 0 when x = 0, which covers every zero denominator).
__device__ __forceinline__ double fmh_metric(uint32_t x, uint64_t nq, uint64_t nr, int k, int metric) {
    if (!x) return 0.0;
    const double dx = (double)x;
    switch (metric) {
        case KMERML_FMH_CONTAINMENT: return dx / (double)nq;
        case KMERML_FMH_MAX_CONTAINMENT: return dx / (double)min(nq, nr);
        case KMERML_FMH_JACCARD: return dx / (double)(nq + nr - x);
        case KMERML_FMH_CONTAINMENT_ANI: return pow(dx / (double)nq, 1.0 / k);
        default: return pow(dx / (double)min(nq, nr), 1.0 / k);
    }
}

__global__ void fmh_metric_kernel(const uint32_t* __restrict__ inter, const uint64_t* __restrict__ q_off, int n_q,
                                  const uint64_t* __restrict__ r_off, int n_r, int k, int metric, float* out32,
                                  double* out64) {
    const uint64_t n = (uint64_t)n_q * n_r;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const int q = (int)(i / n_r), r = (int)(i % n_r);
        const double d = fmh_metric(inter[i], q_off[q + 1] - q_off[q], r_off[r + 1] - r_off[r], k, metric);
        if (out64) out64[i] = d;
        if (out32) out32[i] = (float)d;
    }
}

// Per sketch (a warp each): sum[i] = sum of its abundances, sumsq[i] = sum of their squares (either may be NULL).
__global__ void fmh_abund_sums_kernel(const uint32_t* __restrict__ abund, const uint64_t* __restrict__ off, int n,
                                      unsigned long long* sum, unsigned long long* sumsq) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x / 32);
    for (uint64_t i = blockIdx.x * (uint64_t)(blockDim.x / 32) + threadIdx.x / 32; i < (uint64_t)n; i += warps) {
        unsigned long long s1 = 0, s2 = 0;
        for (uint64_t t = off[i] + lane; t < off[i + 1]; t += 32) {
            const unsigned long long a = abund[t];
            s1 += a;
            s2 += a * a;
        }
        for (int o = 16; o; o >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if (lane == 0) {
            if (sum) sum[i] = s1;
            if (sumsq) sumsq[i] = s2;
        }
    }
}

// Weighted containment x / sum_Q a_Q, or angular similarity 1 - 2 acos(c) / pi with c = min(1, x / (sqrt(qn) sqrt(rn)))
// (x = sum_{Q n R} a_Q a_R, qn and rn the squared norms); 0 when x = 0 or a denominator is 0.  c is 1 whenever
// x^2 = qn rn in integers (Cauchy-Schwarz equality), so proportional abundance vectors give exactly 1 however the
// square roots round.
__global__ void fmh_weighted_metric_kernel(const unsigned long long* __restrict__ num, int n_q, int n_r, int metric,
                                           const unsigned long long* __restrict__ q_den,
                                           const unsigned long long* __restrict__ r_den, float* out32, double* out64) {
    const uint64_t n = (uint64_t)n_q * n_r;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned long long x = num[i], qd = q_den[i / n_r];
        double d = 0.0;
        if (x && qd) {
            if (metric == KMERML_FMH_WEIGHTED_CONTAINMENT) {
                d = (double)x / (double)qd;
            } else {
                const unsigned long long rd = r_den[i % n_r];
                const bool one = x * x == qd * rd && __umul64hi(x, x) == __umul64hi(qd, rd);
                const double c = one ? 1.0 : fmin(1.0, (double)x / (sqrt((double)qd) * sqrt((double)rd)));
                d = 1.0 - 2.0 * acos(c) / 3.141592653589793;
            }
        }
        if (out64) out64[i] = d;
        if (out32) out32[i] = (float)d;
    }
}

size_t fmh_compare_workspace(int n_r) { return (size_t)(n_r + 1) * 8; }

template <bool WEIGHTED>
static int launch_fmh_intersect(const uint64_t* d_qh, const uint64_t* d_q_off, int n_q, const uint64_t* d_rh,
                                const uint64_t* d_r_off, int n_r, int sm_count, void* workspace,
                                std::conditional_t<WEIGHTED, unsigned long long, uint32_t>* d_inter, const uint32_t* d_qa,
                                const uint32_t* d_ra, cudaStream_t s) {
    unsigned long long* prefix = (unsigned long long*)workspace;
    KM_CUDA(cudaMemsetAsync(d_inter, 0, (size_t)n_q * n_r * sizeof(*d_inter), s));
    fmh_chunk_prefix_kernel<<<1, SELECT_THREADS, 0, s>>>(d_r_off, n_r, prefix);
    KM_CUDA(cudaGetLastError());
    KM_CUDA(cudaFuncSetAttribute(fmh_intersect_kernel<WEIGHTED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)FMH_SMEM));
    // three CTAs fit an SM's shared memory; eight rounds of them let the CTAs of long items be balanced by the rest
    fmh_intersect_kernel<WEIGHTED><<<sm_count * 3 * 8, FMH_THREADS, FMH_SMEM, s>>>(d_qh, d_q_off, n_q, d_rh, d_r_off, n_r,
                                                                                prefix, d_inter, d_qa, d_ra);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

size_t fmh_compare_weighted_workspace(int n_q, int n_r) {
    return fmh_compare_workspace(n_r) + (size_t)(2 * n_q + n_r) * 8;
}

int launch_fmh_compare_weighted(const uint64_t* d_qh, const uint64_t* d_q_off, const uint32_t* d_qa, int n_q,
                                const uint64_t* d_rh, const uint64_t* d_r_off, const uint32_t* d_ra, int n_r, int metric,
                                int sm_count, void* workspace, unsigned long long* d_num, float* d_out32, double* d_out64,
                                cudaStream_t s) {
    if (n_q <= 0 || n_r <= 0) return KMERML_OK;
    const bool angular = metric == KMERML_FMH_ANGULAR_SIMILARITY;
    int rc = launch_fmh_intersect<true>(d_qh, d_q_off, n_q, d_rh, d_r_off, n_r, sm_count, workspace, d_num, d_qa,
                                        angular ? d_ra : nullptr, s);
    if (rc || (!d_out32 && !d_out64)) return rc;
    // workspace: the chunk table | sum (weighted containment) or squared norm (angular) of each query | of each reference
    unsigned long long* q_den = (unsigned long long*)workspace + (n_r + 1);
    unsigned long long* r_den = q_den + n_q;
    fmh_abund_sums_kernel<<<(unsigned)std::min<uint64_t>((n_q + 7) / 8, 1ull << 16), 256, 0, s>>>(
        d_qa, d_q_off, n_q, angular ? nullptr : q_den, angular ? q_den : nullptr);
    KM_CUDA(cudaGetLastError());
    if (angular) {
        fmh_abund_sums_kernel<<<(unsigned)std::min<uint64_t>((n_r + 7) / 8, 1ull << 16), 256, 0, s>>>(d_ra, d_r_off, n_r,
                                                                                                  nullptr, r_den);
        KM_CUDA(cudaGetLastError());
    }
    const uint64_t n = (uint64_t)n_q * n_r;
    const uint64_t blocks = std::min<uint64_t>((n + 255) / 256, 1ull << 16);
    fmh_weighted_metric_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_num, n_q, n_r, metric, q_den, r_den, d_out32, d_out64);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

int launch_fmh_compare(const uint64_t* d_qh, const uint64_t* d_q_off, int n_q, const uint64_t* d_rh, const uint64_t* d_r_off,
                       int n_r, int k, int metric, int sm_count, void* workspace, uint32_t* d_inter, float* d_out32,
                       double* d_out64, cudaStream_t s) {
    if (n_q <= 0 || n_r <= 0) return KMERML_OK;
    int rc = launch_fmh_intersect<false>(d_qh, d_q_off, n_q, d_rh, d_r_off, n_r, sm_count, workspace, d_inter, nullptr,
                                         nullptr, s);
    if (rc) return rc;
    if (d_out32 || d_out64) {
        const uint64_t n = (uint64_t)n_q * n_r;
        const uint64_t blocks = std::min<uint64_t>((n + 255) / 256, 1ull << 16);
        fmh_metric_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_inter, d_q_off, n_q, d_r_off, n_r, k, metric, d_out32, d_out64);
        KM_CUDA(cudaGetLastError());
    }
    return KMERML_OK;
}

// ---- gather: greedy, exact split of each query into the references that cover it ---------------------------------
// The host loop is fmh_gather_core (api.cu).  u[q, c] = |Q_{t-1} n R_c| over the candidates c (references with
// |Q n R| >= threshold for some query; u never grows, so no other reference can be picked).
constexpr int GREEDY_THREADS = 256;
constexpr int REMOVE_THREADS = 1024;                  // one CTA holds a whole query: many searches in flight

// flags[r] = 1 when some query shares at least `threshold` hashes with reference r (flags zeroed by the caller).
__global__ void fmh_greedy_flag_kernel(const uint32_t* __restrict__ x, uint64_t n, int n_r, uint32_t threshold,
                                       uint8_t* flags) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        if (x[i] >= threshold) flags[i % n_r] = 1;
}

// Round `round` (< max_matches) of every query still running (pick[q] >= 0), one CTA per query.  Round 0 reads u from
// the prefetched x = |Q n R| (n_q x n_r) through the candidate list; later rounds subtract d = |S_{t-1} n R_c| first.
// The argmax of the key (u << 32) | ~c is the largest u at the smallest candidate index.  The CTA records the match or
// stops the query (pick = -1), and leaves in s_len[q] how many hashes the remove step will assign (0 when stopped).
__global__ void __launch_bounds__(GREEDY_THREADS)
fmh_greedy_select_kernel(uint32_t* u, const uint32_t* __restrict__ d, int n_c, const uint32_t* __restrict__ x, int n_r,
                         const int* __restrict__ cand, const uint64_t* __restrict__ q_off, int round, uint32_t threshold,
                         int max_matches, int* pick, uint32_t* remaining, unsigned long long* s_len, int32_t* n_matches,
                         int32_t* m_ref, uint32_t* m_unique, uint32_t* m_inter, uint32_t* m_rem,
                         unsigned int* n_picked) {
    using Reduce = cub::BlockReduce<unsigned long long, GREEDY_THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    const int q = blockIdx.x;
    if (pick[q] < 0) return;
    uint32_t* row = u + (uint64_t)q * n_c;
    unsigned long long best = 0;
    for (int c = threadIdx.x; c < n_c; c += GREEDY_THREADS) {
        const uint32_t v = round == 0 ? x[(uint64_t)q * n_r + cand[c]] : row[c] - d[(uint64_t)q * n_c + c];
        row[c] = v;
        best = max(best, ((unsigned long long)v << 32) | (uint32_t)~(uint32_t)c);
    }
    best = Reduce(tmp).Reduce(best, cub::Max());
    if (threadIdx.x) return;
    const uint32_t un = (uint32_t)(best >> 32);
    if (un < threshold) {
        pick[q] = -1;
        s_len[q] = 0;
        return;
    }
    const int c = (int)~(uint32_t)best;
    const uint32_t before = round == 0 ? (uint32_t)(q_off[q + 1] - q_off[q]) : remaining[q];
    const uint64_t slot = (uint64_t)q * max_matches + round;
    m_ref[slot] = cand[c];
    m_unique[slot] = un;
    m_inter[slot] = x[(uint64_t)q * n_r + cand[c]];
    m_rem[slot] = remaining[q] = before - un;
    n_matches[q] = round + 1;
    pick[q] = c;
    s_len[q] = un;
    atomicAdd(n_picked, 1u);
}

// S_t of every query that picked candidate c this round: the values of R_c found in Q and not yet assigned, marked
// assigned and written ascending (R_c's order) at s_off[q].  One CTA per query; each value of R_c is a binary search
// in Q.  A count that differs from the select step's u sets *bad.  ABUND: also the query abundances of S_t, written
// beside it, and their sum and sum of squares in slot q * max_matches + round of ab.sum / ab.sumsq.
template <bool ABUND>
__global__ void __launch_bounds__(REMOVE_THREADS)
fmh_greedy_remove_kernel(const uint64_t* __restrict__ qh, const uint64_t* __restrict__ q_off,
                         const uint64_t* __restrict__ ch, const uint64_t* __restrict__ c_off, const int* __restrict__ pick,
                         const unsigned long long* __restrict__ s_off, uint8_t* assigned, uint64_t* s_hashes,
                         unsigned int* bad, GatherAbund ab) {
    using Scan = cub::BlockScan<int, REMOVE_THREADS>;
    __shared__ typename Scan::TempStorage tmp;
    const int q = blockIdx.x;
    const int c = pick[q];
    if (c < 0) return;
    const uint64_t* Q = qh + q_off[q];
    const uint64_t nq = q_off[q + 1] - q_off[q];
    uint8_t* taken = assigned + q_off[q];
    const uint64_t* R = ch + c_off[c];
    const uint64_t nr = c_off[c + 1] - c_off[c];
    uint64_t* out = s_hashes + s_off[q];
    uint64_t written = 0;
    unsigned long long sum = 0, sumsq = 0;            // ABUND: this thread's share
    for (uint64_t base = 0; base < nr; base += REMOVE_THREADS) {
        const uint64_t i = base + threadIdx.x;
        int take = 0;
        uint64_t v = 0;
        uint32_t a = 0;
        if (i < nr) {
            v = R[i];
            uint64_t lo = 0, hi = nq;
            while (lo < hi) {
                const uint64_t mid = (lo + hi) >> 1;
                if (Q[mid] < v) lo = mid + 1; else hi = mid;
            }
            if (lo < nq && Q[lo] == v && !taken[lo]) {
                taken[lo] = 1;
                take = 1;
                if constexpr (ABUND) {
                    a = ab.qa[q_off[q] + lo];
                    sum += a;
                    sumsq += (unsigned long long)a * a;
                }
            }
        }
        int pos, total;
        Scan(tmp).ExclusiveSum(take, pos, total);
        if (take) {
            out[written + pos] = v;
            if constexpr (ABUND) ab.s_abund[s_off[q] + written + pos] = a;
        }
        written += total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && written != s_off[q + 1] - s_off[q]) atomicOr(bad, 1u);
    if constexpr (ABUND) {
        using Reduce = cub::BlockReduce<unsigned long long, REMOVE_THREADS>;
        __shared__ typename Reduce::TempStorage rtmp;
        sum = Reduce(rtmp).Sum(sum);
        __syncthreads();
        sumsq = Reduce(rtmp).Sum(sumsq);
        if (threadIdx.x == 0) {
            const uint64_t slot = (uint64_t)q * ab.max_matches + ab.round;
            ab.sum[slot] = sum;
            ab.sumsq[slot] = sumsq;
        }
    }
}

// The median of the abundances of S_t (sorted per query), for every query that recorded a match this round: the middle
// value, or the mean of the two middle values (exact in float64).
__global__ void fmh_greedy_median_kernel(const uint32_t* __restrict__ sorted, const unsigned long long* __restrict__ s_off,
                                         const int* __restrict__ pick, int n_q, int round, int max_matches, double* median) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_q || pick[q] < 0) return;
    const uint32_t* a = sorted + s_off[q];
    const uint64_t n = s_off[q + 1] - s_off[q];
    median[(uint64_t)q * max_matches + round] = n & 1 ? (double)a[n / 2] : ((double)a[n / 2 - 1] + (double)a[n / 2]) / 2.0;
}

int launch_fmh_greedy_flag(const uint32_t* d_x, int n_q, int n_r, uint32_t threshold, uint8_t* d_flags, cudaStream_t s) {
    const uint64_t n = (uint64_t)n_q * n_r;
    KM_CUDA(cudaMemsetAsync(d_flags, 0, (size_t)n_r, s));
    const uint64_t blocks = std::min<uint64_t>((n + 255) / 256, 1ull << 16);
    fmh_greedy_flag_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_x, n, n_r, threshold, d_flags);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

int launch_fmh_greedy_select(uint32_t* d_u, const uint32_t* d_d, int n_c, const uint32_t* d_x, int n_q, int n_r,
                             const int* d_cand, const uint64_t* d_q_off, int round, uint32_t threshold, int max_matches,
                             int* d_pick, uint32_t* d_remaining, unsigned long long* d_s_len, int32_t* d_n_matches,
                             int32_t* d_ref, uint32_t* d_unique, uint32_t* d_inter, uint32_t* d_rem,
                             unsigned int* d_n_picked, cudaStream_t s) {
    fmh_greedy_select_kernel<<<n_q, GREEDY_THREADS, 0, s>>>(d_u, d_d, n_c, d_x, n_r, d_cand, d_q_off, round, threshold,
                                                           max_matches, d_pick, d_remaining, d_s_len, d_n_matches,
                                                           d_ref, d_unique, d_inter, d_rem, d_n_picked);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

size_t fmh_greedy_scan_temp_bytes(int n_q) {
    size_t t = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, t, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, n_q + 1);
    return t;
}

int launch_fmh_greedy_remove(const uint64_t* d_qh, const uint64_t* d_q_off, int n_q, const uint64_t* d_ch,
                             const uint64_t* d_c_off, const int* d_pick, const unsigned long long* d_s_len,
                             unsigned long long* d_s_off, void* temp, size_t temp_bytes, uint8_t* d_assigned,
                             uint64_t* d_s_hashes, unsigned int* d_bad, const GatherAbund* ab, cudaStream_t s) {
    size_t tb = temp_bytes;
    KM_CUDA(cub::DeviceScan::ExclusiveSum(temp, tb, d_s_len, d_s_off, n_q + 1, s));
    if (ab)
        fmh_greedy_remove_kernel<true><<<n_q, REMOVE_THREADS, 0, s>>>(d_qh, d_q_off, d_ch, d_c_off, d_pick, d_s_off,
                                                                      d_assigned, d_s_hashes, d_bad, *ab);
    else
        fmh_greedy_remove_kernel<false><<<n_q, REMOVE_THREADS, 0, s>>>(d_qh, d_q_off, d_ch, d_c_off, d_pick, d_s_off,
                                                                       d_assigned, d_s_hashes, d_bad, GatherAbund{});
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

size_t fmh_greedy_median_temp_bytes(int n_q, int total) {
    size_t t = 0;
    cub::DeviceSegmentedSort::SortKeys(nullptr, t, (const uint32_t*)nullptr, (uint32_t*)nullptr, total, n_q,
                                       (const unsigned long long*)nullptr, (const unsigned long long*)nullptr);
    return t;
}

int launch_fmh_greedy_median(const GatherAbund& ab, const unsigned long long* d_s_off, const int* d_pick, int n_q,
                             int total, uint32_t* d_sorted, void* temp, size_t temp_bytes, double* d_median,
                             cudaStream_t s) {
    size_t tb = temp_bytes;
    KM_CUDA(cub::DeviceSegmentedSort::SortKeys(temp, tb, (const uint32_t*)ab.s_abund, d_sorted, total, n_q, d_s_off,
                                               d_s_off + 1, s));
    fmh_greedy_median_kernel<<<(n_q + 255) / 256, 256, 0, s>>>(d_sorted, d_s_off, d_pick, n_q, ab.round, ab.max_matches,
                                                               d_median);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

}  // namespace km
