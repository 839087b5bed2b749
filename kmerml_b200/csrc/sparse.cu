// sparse.cu -- k = 15..32: 4^k bins no longer fit a dense histogram, so the windows are emitted as
// 2-bit packed 64-bit keys (+ the byte offset of their last base), radix-sorted and run-length
// reduced into (k-mer, count, first occurrence).  Same window semantics as the dense path
// (kmerml/kmers/generate.py:39-58 of the reference); canonical = min(k-mer, reverse complement).
//
// Round 1: the sort and the segmented reductions are CUB library calls (the toolkit's own headers);
// the emitter is the shared carry-free walker with 64-bit state.
#include <cub/cub.cuh>
#include <thrust/iterator/constant_iterator.h>

#include "sparse_walk.cuh"

namespace km {

// Every window to the caller's arrays.  Fast lanes: the windows of a warp's 32 chunks are written window-index-major
// with ONE cursor reservation per warp and tile, so the 8-byte key stores and 4-byte offset stores are contiguous
// across the lanes.  Byte walker: one reservation per warp instead of one per window.
struct WindowSink {
    uint64_t* keys;
    uint32_t* ends;
    unsigned long long* cursor;
    uint64_t cap;
    struct Lanes {                // a warp's reservation for its fast lanes' windows
        unsigned long long base;
        unsigned n_fast, rank, rank32;
    };
    __device__ __forceinline__ Lanes fast_begin(bool fast, unsigned fast_mask, unsigned n31_mask, int lane) const {
        Lanes l;
        const unsigned total = 32u * __popc(fast_mask) - __popc(n31_mask);
        l.base = 0;
        if (lane == 0) l.base = atomicAdd(cursor, (unsigned long long)total);
        l.base = __shfl_sync(0xffffffffu, l.base, 0);
        const unsigned below = fast_mask & ((1u << lane) - 1u);
        l.rank = __popc(below);
        l.n_fast = __popc(fast_mask);
        l.rank32 = __popc(below & ~n31_mask);
        return l;
    }
    __device__ __forceinline__ void fast_window(const Lanes& l, int j, uint64_t key, uint64_t pos) const {
        const unsigned long long slot = l.base + (j < 31 ? (unsigned long long)j * l.n_fast + l.rank
                                                         : 31ull * l.n_fast + l.rank32);
        if (slot < cap) {
            keys[slot] = key;
            ends[slot] = (uint32_t)pos;
        }
    }
    __device__ __forceinline__ void window(uint64_t key, uint64_t pos) const {
        const unsigned active = __activemask();
        const int lane = threadIdx.x & 31;
        const int leader = __ffs(active) - 1;
        unsigned long long b = 0;
        if (lane == leader) b = atomicAdd(cursor, (unsigned long long)__popc(active));
        b = __shfl_sync(active, b, leader);
        const unsigned long long slot = b + __popc(active & ((1u << lane) - 1u));
        if (slot < cap) {
            keys[slot] = key;
            ends[slot] = (uint32_t)pos;
        }
    }
};

__global__ void sparse_setup_kernel(const uint8_t* __restrict__ buf, uint64_t nbytes, GenomeDev* gd, Slice* slices,
                                    int n_slices) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        gd->file_lo = 0;
        gd->lo = first_header(buf, 0, nbytes);       // text before the first header line is ignored
        gd->hi = nbytes;
    }
    if (i <= n_slices) {                             // entry n_slices = scratch of launch_slice_headers
        Slice sl;
        sl.genome = 0; sl.prev_ok = 0; sl.prev16 = 0; sl.tile0 = 0; sl.hdr_until = 0;
        sl.begin = (uint64_t)i * SPARSE_TILE * SPARSE_TILES_PER_SLICE;
        sl.end = sl.begin + (uint64_t)SPARSE_TILE * SPARSE_TILES_PER_SLICE;
        sl.line_start = 0; sl.scan_last = 0;
        slices[i] = sl;
    }
}

__global__ void __launch_bounds__(SPARSE_THREADS)
sparse_emit_kernel(const uint8_t* __restrict__ buf, const GenomeDev* __restrict__ gds, const Slice* __restrict__ slices,
                   SparseParams P, uint64_t* keys, uint32_t* ends, unsigned long long* cursor, uint64_t cap) {
    const Slice sl = slices[blockIdx.x];
    const GenomeDev gd = gds[0];
    WindowSink sink;
    sink.keys = keys; sink.ends = ends; sink.cursor = cursor; sink.cap = cap;
    walk_sparse_slice(buf, gd, sl, P, sink);
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ src, uint32_t* dst, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}

struct CountFirst {               // count in the high word, first (smallest) offset in the low word
    __host__ __device__ __forceinline__ unsigned long long operator()(unsigned long long a, unsigned long long b) const {
        const unsigned long long cnt = (a >> 32) + (b >> 32);
        const unsigned long long fa = a & 0xFFFFFFFFull, fb = b & 0xFFFFFFFFull;
        return (cnt << 32) | (fa < fb ? fa : fb);
    }
};
struct OneWindow {                // a sorted window's end offset -> (count 1, first = that offset)
    __host__ __device__ __forceinline__ unsigned long long operator()(uint32_t end) const { return (1ull << 32) | end; }
};

__global__ void unpack_count_first_kernel(const unsigned long long* __restrict__ in, uint64_t n, uint32_t* counts,
                                          uint32_t* first) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    counts[i] = (uint32_t)(in[i] >> 32);
    if (first) first[i] = (uint32_t)in[i];
}

// Output iterator of the fused segmented reduction: a packed (count, first) aggregate goes straight into the
// caller's two arrays.
struct SplitCountFirst {
    uint32_t* counts;
    uint32_t* first;              // may be null
    struct Ref {
        uint32_t* c;
        uint32_t* f;
        __host__ __device__ __forceinline__ Ref& operator=(unsigned long long v) {
            *c = (uint32_t)(v >> 32);
            if (f) *f = (uint32_t)v;
            return *this;
        }
    };
    using iterator_category = std::random_access_iterator_tag;
    using value_type = unsigned long long;
    using difference_type = ptrdiff_t;
    using pointer = void;
    using reference = Ref;
    __host__ __device__ __forceinline__ Ref operator*() const { return Ref{counts, first}; }
    __host__ __device__ __forceinline__ Ref operator[](difference_type i) const { return Ref{counts + i, first ? first + i : nullptr}; }
    __host__ __device__ __forceinline__ SplitCountFirst operator+(difference_type i) const {
        return SplitCountFirst{counts + i, first ? first + i : nullptr};
    }
};

// distinct keys of a sorted array = 1 + the positions whose key differs from the one before
__global__ void __launch_bounds__(256)
count_boundaries_kernel(const uint64_t* __restrict__ keys, uint64_t n, unsigned long long* out) {
    unsigned long long mine = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        mine += (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(out, mine);
}

struct SparseWork {
    uint64_t* keys_a;
    uint64_t* keys_b;
    uint32_t* ends_a;
    uint32_t* ends_b;
    unsigned long long* cursor;
    unsigned long long* n_runs;
    GenomeDev* genome;
    Slice* slices;
    void* temp;
    size_t temp_bytes;
};

// Layout of the workspace for `cap` windows; returns the total number of bytes.
size_t sparse_workspace(uint64_t cap, uint64_t nbytes, SparseWork* w, uint8_t* base) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        uint8_t* p = base ? base + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return p;
    };
    SparseWork local;
    local.keys_a = (uint64_t*)take(cap * 8);
    local.keys_b = (uint64_t*)take(cap * 8);
    local.ends_a = (uint32_t*)take(cap * 4);
    local.ends_b = (uint32_t*)take(cap * 4);
    local.cursor = (unsigned long long*)take(256);
    local.n_runs = (unsigned long long*)take(256);
    local.genome = (GenomeDev*)take(256);
    // one slice entry per 128 KB of the whole file + scratch
    local.slices = (Slice*)take((nbytes / ((uint64_t)SPARSE_TILE * SPARSE_TILES_PER_SLICE) + 3) * sizeof(Slice));
    size_t t1 = 0, t2 = 0, t3 = 0;
    cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
    cub::DoubleBuffer<uint32_t> dv(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, t1, dk, dv, (uint64_t)cap, 0, 64);
    {
        cub::TransformInputIterator<unsigned long long, OneWindow, const uint32_t*> vin((const uint32_t*)nullptr, OneWindow());
        cub::DeviceReduce::ReduceByKey(nullptr, t2, (const uint64_t*)nullptr, (uint64_t*)nullptr, vin,
                                       SplitCountFirst{nullptr, nullptr}, (unsigned long long*)nullptr, CountFirst(),
                                       (uint64_t)cap);
    }
    (void)t3;
    local.temp_bytes = std::max(t1, std::max(t2, t3));
    local.temp = take(local.temp_bytes);
    if (w) *w = local;
    return off;
}

// The reduced result (distinct k-mers in `uniq`, their counts in `runs`) to the caller's buffers; the first
// offsets are the minimum end offset of every run of the sorted windows.
static int sparse_copy_out(const SparseWork& w, uint64_t* sorted_keys, uint32_t* sorted_ends, uint64_t* uniq, uint32_t* runs,
                           uint64_t n, uint64_t nu, uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out,
                           cudaStream_t s) {
    // ONE segmented reduction over the sorted windows: distinct k-mers to the caller's key array, (run length, smallest
    // end offset) through a splitting output iterator to its count / first-offset arrays
    (void)uniq; (void)runs; (void)nu;
    cub::TransformInputIterator<unsigned long long, OneWindow, const uint32_t*> vin(sorted_ends, OneWindow());
    size_t tb = w.temp_bytes;
    KM_CUDA(cub::DeviceReduce::ReduceByKey(w.temp, tb, (const uint64_t*)sorted_keys, d_keys_out, vin,
                                           SplitCountFirst{d_counts_out, d_first_out}, w.n_runs, CountFirst(), (uint64_t)n, s));
    KM_CUDA(cudaStreamSynchronize(s));
    return KMERML_OK;
}

// Emit the windows of the byte range into w.keys_a / w.ends_a; *h_windows receives their number.
static int sparse_emit_phase(const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin, uint64_t range_end, int k,
                             int min_rec, bool canonical, const SparseWork& w, uint64_t cap, uint64_t* h_windows,
                             cudaStream_t s) {
    SparseParams P;
    P.k = k;
    P.min_rec = min_rec;
    P.canonical = canonical ? 1 : 0;
    P.mask = k >= 32 ? ~0ull : ((1ull << (2 * k)) - 1ull);
    KM_CUDA(cudaMemsetAsync(w.cursor, 0, 8, s));
    *h_windows = 0;
    if (!nbytes) return KMERML_OK;
    const uint64_t slice_bytes = (uint64_t)SPARSE_TILE * SPARSE_TILES_PER_SLICE;
    const int n_slices = (int)((nbytes + slice_bytes - 1) / slice_bytes);
    sparse_setup_kernel<<<(n_slices + 1 + 127) / 128, 128, 0, s>>>(d_fasta, nbytes, w.genome, w.slices, n_slices);
    KM_CUDA(cudaGetLastError());
    if (int rc = launch_slice_headers(d_fasta, w.genome, w.slices, n_slices, s)) return rc;
    // the header state of every slice start is settled over the whole file; only the slices of the
    // requested byte range (whole slices: the multi-GPU unit) emit their windows
    const int s0 = (int)std::min<uint64_t>(range_begin / slice_bytes, (uint64_t)n_slices);
    const int s1 = (int)std::min<uint64_t>((range_end + slice_bytes - 1) / slice_bytes, (uint64_t)n_slices);
    if (s1 > s0) {
        sparse_emit_kernel<<<s1 - s0, SPARSE_THREADS, 0, s>>>(d_fasta, w.genome, w.slices + s0, P, w.keys_a, w.ends_a,
                                                              w.cursor, cap);
        KM_CUDA(cudaGetLastError());
    }
    unsigned long long n = 0;
    KM_CUDA(cudaMemcpyAsync(&n, w.cursor, 8, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    *h_windows = n;
    if (n > cap) {
        set_error("internal: sparse window capacity exceeded");
        return KMERML_ERR_RANGE;
    }
    return KMERML_OK;
}

// Sort the n windows in w.keys_a / w.ends_a by bits [0, sort_bits) of the key and reduce them.
static int sparse_sort_reduce_phase(const SparseWork& w, uint64_t n, int sort_bits, uint64_t* d_keys_out, uint32_t* d_counts_out,
                                    uint32_t* d_first_out, uint64_t out_cap, uint64_t* h_unique, SparsePending* pending,
                                    cudaStream_t s) {
    *h_unique = 0;
    if (!n) return KMERML_OK;
    KM_CUDA(cudaMemsetAsync(w.n_runs, 0, 8, s));
    cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
    cub::DoubleBuffer<uint32_t> dv(w.ends_a, w.ends_b);
    size_t tb = w.temp_bytes;
    // radix sort is stable and the emission order is arbitrary, so the first occurrence is the
    // MIN end offset of each run, not its first element
    KM_CUDA(cub::DeviceRadixSort::SortPairs(w.temp, tb, dk, dv, (uint64_t)n, 0, sort_bits, s));
    uint64_t* sorted_keys = dk.Current();
    uint32_t* sorted_ends = dv.Current();
    uint64_t* uniq = dk.Alternate();
    uint32_t* runs = dv.Alternate();
    // number of distinct k-mers first (one read of the sorted keys): the caller's buffers may be too small
    count_boundaries_kernel<<<148 * 8, 256, 0, s>>>(sorted_keys, (uint64_t)n, w.n_runs);
    KM_CUDA(cudaGetLastError());
    unsigned long long nu = 0;
    KM_CUDA(cudaMemcpyAsync(&nu, w.n_runs, 8, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    *h_unique = nu;
    if (pending) {
        pending->sorted_keys = sorted_keys; pending->sorted_ends = sorted_ends; pending->uniq = uniq; pending->runs = runs;
        pending->n = n; pending->nu = nu; pending->valid = true;
    }
    if (nu > out_cap) return KMERML_OK;             // caller sizes its outputs and fetches (kmerml_sparse_fetch)
    return sparse_copy_out(w, sorted_keys, sorted_ends, uniq, runs, n, nu, d_keys_out, d_counts_out, d_first_out, s);
}

// Emits, sorts and reduces.  On return (after a stream sync) *h_windows / *h_unique are valid; when
// *h_unique > out_cap nothing was written to the outputs (kmerml_sparse_fetch copies them out later).
int run_sparse(const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin, uint64_t range_end, int k, int min_rec,
               bool canonical, const SparseWork& w, uint64_t cap, uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
               uint64_t* h_unique, uint64_t* h_windows, SparsePending* pending, cudaStream_t s) {
    if (pending) pending->valid = false;
    *h_unique = 0;
    if (int rc = sparse_emit_phase(d_fasta, nbytes, range_begin, range_end, k, min_rec, canonical, w, cap, h_windows, s)) return rc;
    return sparse_sort_reduce_phase(w, *h_windows, 2 * k, d_keys_out, d_counts_out, d_first_out, out_cap, h_unique, pending, s);
}

// ---- multi-GPU, raw routing: a rank emits the windows of its byte range, groups them by the rank that owns
// their key range (ONE radix pass over the top owner_bits of the k-mer) and reports how many each owner gets; after
// the exchange every rank sorts and reduces what it received ONCE (kmerml_reduce_sparse_windows).
__global__ void owner_bounds_kernel(const uint64_t* __restrict__ keys, uint64_t n, int shift, int n_owners,
                                    unsigned long long* bounds /* n_owners + 1 */) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n_owners) return;
    // first index whose owner (key >> shift) is >= r: the keys are grouped by owner, ascending
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if ((keys[mid] >> shift) < (uint64_t)r) lo = mid + 1; else hi = mid;
    }
    bounds[r] = lo;
}

int run_sparse_emit_by_owner(void* workspace, const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin,
                             uint64_t range_end, int k, int min_rec, bool canonical, int owner_bits, uint64_t cap,
                             uint64_t* d_keys_out, uint32_t* d_ends_out, uint64_t out_cap, uint64_t* h_windows,
                             uint64_t* h_owner_counts, cudaStream_t s) {
    SparseWork w;
    sparse_workspace(cap, nbytes, &w, (uint8_t*)workspace);
    const int n_owners = 1 << owner_bits;
    for (int r = 0; r < n_owners; r++) h_owner_counts[r] = 0;
    if (int rc = sparse_emit_phase(d_fasta, nbytes, range_begin, range_end, k, min_rec, canonical, w, cap, h_windows, s)) return rc;
    const uint64_t n = *h_windows;
    if (!n || n > out_cap) return KMERML_OK;
    uint64_t* keys = w.keys_a;
    uint32_t* ends = w.ends_a;
    if (owner_bits > 0) {
        cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
        cub::DoubleBuffer<uint32_t> dv(w.ends_a, w.ends_b);
        size_t tb = w.temp_bytes;
        KM_CUDA(cub::DeviceRadixSort::SortPairs(w.temp, tb, dk, dv, n, 2 * k - owner_bits, 2 * k, s));
        keys = dk.Current();
        ends = dv.Current();
    }
    unsigned long long* d_bounds = w.n_runs;                      // (256 bytes: up to 31 owners + 1)
    owner_bounds_kernel<<<1, 64, 0, s>>>(keys, n, 2 * k - owner_bits, n_owners, d_bounds);
    KM_CUDA(cudaGetLastError());
    unsigned long long h_bounds[33];
    KM_CUDA(cudaMemcpyAsync(h_bounds, d_bounds, (size_t)(n_owners + 1) * 8, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaMemcpyAsync(d_keys_out, keys, n * 8, cudaMemcpyDeviceToDevice, s));
    KM_CUDA(cudaMemcpyAsync(d_ends_out, ends, n * 4, cudaMemcpyDeviceToDevice, s));
    KM_CUDA(cudaStreamSynchronize(s));
    for (int r = 0; r < n_owners; r++) h_owner_counts[r] = h_bounds[r + 1] - h_bounds[r];
    return KMERML_OK;
}

int run_sparse_reduce_windows(void* workspace, int sort_bits, const uint64_t* d_keys, const uint32_t* d_ends, uint64_t n,
                              uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                              uint64_t* h_unique, SparsePending* pending, cudaStream_t s) {
    if (pending) pending->valid = false;
    *h_unique = 0;
    if (!n) return KMERML_OK;
    SparseWork w;
    sparse_workspace(n, 0, &w, (uint8_t*)workspace);
    KM_CUDA(cudaMemcpyAsync(w.keys_a, d_keys, n * 8, cudaMemcpyDeviceToDevice, s));
    KM_CUDA(cudaMemcpyAsync(w.ends_a, d_ends, n * 4, cudaMemcpyDeviceToDevice, s));
    return sparse_sort_reduce_phase(w, n, sort_bits, d_keys_out, d_counts_out, d_first_out, out_cap, h_unique, pending, s);
}

int sparse_fetch(void* workspace, uint64_t cap, uint64_t nbytes, const SparsePending& p, uint64_t* d_keys_out,
                 uint32_t* d_counts_out, uint32_t* d_first_out, cudaStream_t s) {
    SparseWork w;
    sparse_workspace(cap, nbytes, &w, (uint8_t*)workspace);
    return sparse_copy_out(w, p.sorted_keys, p.sorted_ends, p.uniq, p.runs, p.n, p.nu, d_keys_out, d_counts_out,
                           d_first_out, s);
}

size_t sparse_workspace_bytes(uint64_t cap, uint64_t nbytes) { return sparse_workspace(cap, nbytes, nullptr, nullptr); }

int run_sparse_in(void* workspace, const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin, uint64_t range_end,
                  int k, int min_rec, bool canonical, uint64_t cap, uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                  uint64_t* h_unique, uint64_t* h_windows, SparsePending* pending, cudaStream_t s) {
    SparseWork w;
    sparse_workspace(cap, nbytes, &w, (uint8_t*)workspace);
    return run_sparse(d_fasta, nbytes, range_begin, range_end, k, min_rec, canonical, w, cap, d_keys_out, d_counts_out, d_first_out, out_cap,
                      h_unique, h_windows, pending, s);
}

// ---- merge of partial results (multi-GPU: every rank receives the (k-mer, count, first) triples of its
// key range from all ranks): sort by k-mer, add the counts, keep the smallest first offset.
__global__ void pack_count_first_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ first,
                                        uint64_t n, unsigned long long* out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = ((unsigned long long)counts[i] << 32) | (first ? first[i] : 0xFFFFFFFFu);
}

struct MergeWork {
    uint64_t* keys_a;
    uint64_t* keys_b;
    unsigned long long* vals_a;
    unsigned long long* vals_b;
    unsigned long long* n_runs;
    void* temp;
    size_t temp_bytes;
};

static size_t merge_layout(uint64_t n, MergeWork* w, uint8_t* base) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        uint8_t* p = base ? base + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return p;
    };
    MergeWork l;
    l.keys_a = (uint64_t*)take(n * 8);
    l.keys_b = (uint64_t*)take(n * 8);
    l.vals_a = (unsigned long long*)take(n * 8);
    l.vals_b = (unsigned long long*)take(n * 8);
    l.n_runs = (unsigned long long*)take(256);
    size_t t1 = 0, t2 = 0;
    cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
    cub::DoubleBuffer<unsigned long long> dv(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, t1, dk, dv, (uint64_t)n, 0, 64);
    cub::DeviceReduce::ReduceByKey(nullptr, t2, (uint64_t*)nullptr, (uint64_t*)nullptr, (unsigned long long*)nullptr,
                                   (unsigned long long*)nullptr, (unsigned long long*)nullptr, CountFirst(), (uint64_t)n);
    l.temp_bytes = std::max(t1, t2);
    l.temp = take(l.temp_bytes);
    if (w) *w = l;
    return off;
}

size_t merge_workspace_bytes(uint64_t n) { return merge_layout(n, nullptr, nullptr); }

int run_merge_sparse(void* workspace, int k, const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first,
                     uint64_t n, uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                     uint64_t* h_unique, cudaStream_t s) {
    *h_unique = 0;
    if (!n) return KMERML_OK;
    MergeWork w;
    merge_layout(n, &w, (uint8_t*)workspace);
    KM_CUDA(cudaMemcpyAsync(w.keys_a, d_keys, n * 8, cudaMemcpyDeviceToDevice, s));
    pack_count_first_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_counts, d_first, n, w.vals_a);
    KM_CUDA(cudaGetLastError());
    cub::DoubleBuffer<uint64_t> dk(w.keys_a, w.keys_b);
    cub::DoubleBuffer<unsigned long long> dv(w.vals_a, w.vals_b);
    size_t tb = w.temp_bytes;
    KM_CUDA(cub::DeviceRadixSort::SortPairs(w.temp, tb, dk, dv, (uint64_t)n, 0, 2 * k, s));
    tb = w.temp_bytes;
    KM_CUDA(cudaMemsetAsync(w.n_runs, 0, 8, s));
    KM_CUDA(cub::DeviceReduce::ReduceByKey(w.temp, tb, dk.Current(), dk.Alternate(), dv.Current(), dv.Alternate(),
                                           w.n_runs, CountFirst(), (uint64_t)n, s));
    unsigned long long nu = 0;
    KM_CUDA(cudaMemcpyAsync(&nu, w.n_runs, 8, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    *h_unique = nu;
    if (nu > out_cap) return KMERML_OK;                 // caller re-sizes and calls again
    KM_CUDA(cudaMemcpyAsync(d_keys_out, dk.Alternate(), nu * 8, cudaMemcpyDeviceToDevice, s));
    unpack_count_first_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, s>>>(dv.Alternate(), nu, d_counts_out, d_first_out);
    KM_CUDA(cudaGetLastError());
    KM_CUDA(cudaStreamSynchronize(s));
    return KMERML_OK;
}

}  // namespace km
