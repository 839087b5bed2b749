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

int launch_sketch_select(const SketchGenome* d_sg, const int* d_active, int n_active, int* d_seg, int n_items,
                         const uint64_t* d_regions, uint64_t* d_sorted, void* temp, size_t temp_bytes, int sketch_size,
                         uint64_t* d_sketches, uint64_t stride, uint32_t* d_filled, uint32_t* d_status, cudaStream_t s) {
    if (n_active <= 0) return KMERML_OK;
    int* seg_begin = d_seg;
    int* seg_end = d_seg + n_active;
    sketch_segments_kernel<<<(n_active + 255) / 256, 256, 0, s>>>(d_sg, d_active, n_active, seg_begin, seg_end);
    KM_CUDA(cudaGetLastError());
    size_t tb = temp_bytes;
    KM_CUDA(cub::DeviceSegmentedSort::SortKeys(temp, tb, d_regions, d_sorted, n_items, n_active, (const int*)seg_begin,
                                               (const int*)seg_end, s));
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

}  // namespace km
