// api.cu -- the C-ABI of libkmerml_b200.so (include/kmerml_b200.h) and the host
// orchestration of the dense counting path.  No torch types, no CPU fallback.
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "internal.h"

namespace km {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    return KMERML_ERR_CUDA;
}
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return KMERML_OK;
        if (p) KM_CUDA(cudaFree(p));
        p = nullptr;
        cap = 0;
        size_t want = std::max<size_t>(bytes, 256);
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            (void)cudaGetLastError();
            return fail(KMERML_ERR_NOMEM, "device allocation of " + std::to_string(want) + " bytes failed");
        }
        cap = want;
        return KMERML_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return KMERML_OK;
        if (p) KM_CUDA(cudaFreeHost(p));
        p = nullptr;
        cap = 0;
        size_t want = std::max<size_t>(bytes, 4096);
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            (void)cudaGetLastError();
            return fail(KMERML_ERR_NOMEM, "pinned allocation of " + std::to_string(want) + " bytes failed");
        }
        cap = want;
        return KMERML_OK;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// Tables + scratch used by one in-flight counting call.
struct Workspace {
    DevBuf tables;      // offsets | GenomeDev | GenomeStats | Slice[]
    DevBuf scratch;     // pass-through cascade levels
    DevBuf part;        // partition path: bucket-sorted payloads + per-tile offset tables
    DevBuf misc;        // record scan counter, Gram matrix
    PinBuf staging;     // host image of offsets + slices
    cudaEvent_t staging_free = nullptr;
    // host-path slot buffers
    DevBuf fasta, counts, freq, totals;
    DevBuf wire;        // narrow D2H: bytes of the levels k >= 10 | exception count | exception list
    PinBuf wire_host;   // ... and its pinned host image
    cudaStream_t stream = nullptr;
    void release() {
        tables.release(); scratch.release(); part.release(); misc.release(); staging.release();
        fasta.release(); counts.release(); freq.release(); totals.release(); wire.release(); wire_host.release();
        if (staging_free) cudaEventDestroy(staging_free);
        if (stream) cudaStreamDestroy(stream);
        staging_free = nullptr;
        stream = nullptr;
    }
};

}  // namespace km

struct ProfRec {
    int kind;                 // 0 count, 1 cascade, 2 finalize, 3 other, 4 partition, 5 bucket
    cudaEvent_t a, b;
};

struct kmerml_ctx {
    int device = 0;
    int sm_count = 148;
    km::Workspace ws[8];                          // [0]: device-resident calls; [0..n): the host pipeline's slots
    int host_slots = 6;                           // (measured: 2 slots 29.8, 3: 39.4, 4: 34.9, 6: 45.3, 8: 44.7 Gbp/s for the compact call, 60 C2 genomes)
    km::SparsePending sparse_pending;             // kmerml_count_sparse -> kmerml_sparse_fetch
    km::DevBuf fmh_kept;                          // kmerml_fmh_batch -> kmerml_fmh_fetch: the kept values of every round,
    km::DevBuf fmh_index;                         // where each genome's begin there | the CSR offsets
    km::DevBuf fmh_abund;                         // KMERML_FLAG_FMH_ABUNDANCE: the abundances, parallel to fmh_kept
    int fmh_n = -1;                               // genomes of that result (< 0: none)
    bool fmh_has_abund = false;                   // that result was made with KMERML_FLAG_FMH_ABUNDANCE
    uint64_t fmh_total = 0;
    km::HostPool* host_pool = nullptr;            // host threads that widen the narrow D2H format
    cudaStream_t last_stream = nullptr;           // ws[0] is scratch shared by every device-resident call: a call on
    bool last_stream_valid = false;               // another stream than the one before waits for that one (order_stream)
    cudaEvent_t order_ev = nullptr;
    uint64_t max_group_payload = 12ull << 30;     // partition path: payload bytes one group of genomes may take
    // measurement hooks
    bool profiling = false;
    uint64_t launches = 0, count_launches = 0;
    std::vector<ProfRec> recs;
    std::vector<cudaEvent_t> pool;
    double ms[6] = {0, 0, 0, 0, 0, 0};
};

namespace km {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The scratch buffers of ws[0] are reused from call to call.  Calls on ONE stream are ordered by the stream; a call on
// another stream than the previous one first waits for what that one still has in flight.
static int order_stream(kmerml_ctx* ctx, cudaStream_t s) {
    if (ctx->last_stream_valid && ctx->last_stream != s) {
        if (!ctx->order_ev) KM_CUDA(cudaEventCreateWithFlags(&ctx->order_ev, cudaEventDisableTiming));
        if (cudaEventRecord(ctx->order_ev, ctx->last_stream) == cudaSuccess) {
            KM_CUDA(cudaStreamWaitEvent(s, ctx->order_ev, 0));
        } else {                                    // the caller destroyed that stream: its work is done or abandoned
            (void)cudaGetLastError();
            KM_CUDA(cudaDeviceSynchronize());
        }
    }
    ctx->last_stream = s;
    ctx->last_stream_valid = true;
    return KMERML_OK;
}

// Brackets a group of launches with events when profiling is on; always counts launches.
struct Prof {
    kmerml_ctx* ctx;
    cudaStream_t s;
    int kind;
    cudaEvent_t a = nullptr, b = nullptr;
    Prof(kmerml_ctx* c, cudaStream_t st, int k, int n_launches) : ctx(c), s(st), kind(k) {
        ctx->launches += (uint64_t)n_launches;
        if (k == 0 || k == 4) ctx->count_launches += (uint64_t)n_launches;
        if (!ctx->profiling) return;
        a = take();
        b = take();
        if (a && b) cudaEventRecord(a, s);
    }
    cudaEvent_t take() {
        cudaEvent_t e = nullptr;
        if (!ctx->pool.empty()) { e = ctx->pool.back(); ctx->pool.pop_back(); return e; }
        if (cudaEventCreate(&e) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
        return e;
    }
    ~Prof() {
        if (!a || !b) return;
        cudaEventRecord(b, s);
        ctx->recs.push_back({kind, a, b});
    }
};

// The tables the host builds for one call: 256-byte-aligned blocks at the same offsets in ws.staging, where the host
// fills them, and in ws.tables, where the kernels read them.  take() every block, open(), then fill() and upload().
struct Tables {
    Workspace& ws;
    size_t size = 0;
    std::vector<std::pair<size_t, size_t>> filled;          // (offset, bytes) of the blocks to upload
    size_t take(size_t bytes) {
        const size_t at = size;
        size += align_up(bytes, 256);
        return at;
    }
    int open() {
        int rc = ws.tables.ensure(size);
        if (!rc) rc = ws.staging.ensure(size);
        if (rc) return rc;
        if (!ws.staging_free) KM_CUDA(cudaEventCreateWithFlags(&ws.staging_free, cudaEventDisableTiming));
        KM_CUDA(cudaEventSynchronize(ws.staging_free));     // the previous call's upload has left the staging buffer
        return KMERML_OK;
    }
    template <class T> T* dev(size_t at) const { return (T*)((uint8_t*)ws.tables.p + at); }
    template <class T> T* host(size_t at) const { return (T*)((uint8_t*)ws.staging.p + at); }
    // the host image of `bytes` bytes at `at`, uploaded by the next upload()
    template <class T> T* fill(size_t at, size_t bytes) {
        filled.push_back({at, bytes});
        return host<T>(at);
    }
    int upload(cudaStream_t s) {                             // the filled blocks, in layout order
        std::sort(filled.begin(), filled.end());
        for (const auto& b : filled)
            KM_CUDA(cudaMemcpyAsync(dev<uint8_t>(b.first), host<uint8_t>(b.first), b.second, cudaMemcpyHostToDevice, s));
        filled.clear();
        KM_CUDA(cudaEventRecord(ws.staging_free, s));
        return KMERML_OK;
    }
};

// The slice table of a walk over the FASTA bytes: every walker's CTAs take their work from one.  Genome g's bytes
// [offsets[g], offsets[g + 1]), clipped to [range_begin, range_end) when range_end != 0, are cut at absolute multiples
// of slice_bytes[g] (0: no slices for g).  A slice's end is clipped to the range; its begin never lies before the tile
// (`tile` bytes) that holds the genome's first walked byte, so no CTA walks the empty tiles below a genome.  The slices
// are in buffer order, genome g's are [first[g], first[g + 1]), and the last entry is the scratch entry of
// launch_slice_headers.
static int plan_slices(const uint64_t* offsets, int n, const uint64_t* slice_bytes, uint64_t tile, uint64_t range_begin,
                       uint64_t range_end, std::vector<Slice>& slices, std::vector<uint32_t>& first) {
    slices.clear();
    first.resize(n + 1);
    for (int g = 0; g < n; g++) {
        first[g] = (uint32_t)slices.size();
        const uint64_t sb = slice_bytes[g];
        uint64_t lo = offsets[g], hi = offsets[g + 1];
        if (range_end) { lo = std::max(lo, range_begin); hi = std::min(hi, range_end); }
        if (!sb || lo >= hi) continue;
        const uint64_t b0 = lo / sb, b1 = (hi - 1) / sb;
        if (slices.size() + (b1 - b0 + 1) > 0x7fffffffull) return fail(KMERML_ERR_RANGE, "too many slices");
        for (uint64_t b = b0; b <= b1; b++) {
            Slice sl{};
            sl.genome = (uint32_t)g;
            sl.begin = std::max(b * sb, lo / tile * tile);
            sl.end = range_end ? std::min((b + 1) * sb, range_end) : (b + 1) * sb;
            slices.push_back(sl);
        }
    }
    first[n] = (uint32_t)slices.size();
    slices.push_back(Slice{});
    return KMERML_OK;
}

// A slice table in a call's Tables: the blocks offsets | genome descriptors | stats, and the slices (+ the scratch
// entry) in a block of their own, which a caller may lay out after its own tables.
struct Walk {
    size_t offsets, genomes, stats, slices = 0;
    int n_genomes, n_slices = 0;
    Walk(Tables& t, int n)
        : offsets(t.take((size_t)(n + 1) * 8)), genomes(t.take((size_t)n * sizeof(GenomeDev))),
          stats(t.take((size_t)n * sizeof(GenomeStats))), n_genomes(n) {}
    void take_slices(Tables& t, size_t max_slices) { slices = t.take((max_slices + 1) * sizeof(Slice)); }
};

// Puts a walk on the device: uploads every block filled so far, plus the genome offsets when `h_offsets` is given
// (then launch_prologue fills the genome descriptors and zeroes the stats) and the planned slices when `plan` is given
// (then the slice-table kernels settle the header state at every slice start).
static int put_walk(Tables& t, Walk& w, const uint8_t* d_fasta, const uint64_t* h_offsets, const std::vector<Slice>* plan,
                    cudaStream_t s) {
    if (h_offsets) memcpy(t.fill<uint64_t>(w.offsets, (size_t)(w.n_genomes + 1) * 8), h_offsets, (size_t)(w.n_genomes + 1) * 8);
    if (plan) {
        memcpy(t.fill<Slice>(w.slices, plan->size() * sizeof(Slice)), plan->data(), plan->size() * sizeof(Slice));
        w.n_slices = (int)plan->size() - 1;
    }
    int rc = t.upload(s);
    if (!rc && h_offsets)
        rc = launch_prologue(d_fasta, t.dev<uint64_t>(w.offsets), t.dev<GenomeDev>(w.genomes), t.dev<GenomeStats>(w.stats),
                             w.n_genomes, s);
    if (!rc && plan) rc = launch_slice_headers(d_fasta, t.dev<GenomeDev>(w.genomes), t.dev<Slice>(w.slices), w.n_slices, s);
    return rc;
}

// The walk of ONE genome that fills [0, nbytes) of the buffer, in slices of `slice_bytes` (first occurrence, encode,
// sparse), on the device.  No bytes: no slices, nothing launched.
struct DevWalk {
    const GenomeDev* genomes = nullptr;
    const Slice* slices = nullptr;
    int n_slices = 0;
};
static int put_single_walk(Workspace& ws, const uint8_t* d_fasta, uint64_t nbytes, uint64_t slice_bytes, uint64_t tile,
                           cudaStream_t s, DevWalk* out) {
    if (!nbytes) return KMERML_OK;
    const uint64_t offs[2] = {0, nbytes};
    std::vector<Slice> plan;
    std::vector<uint32_t> first;
    int rc = plan_slices(offs, 1, &slice_bytes, tile, 0, 0, plan, first);
    if (rc) return rc;
    Tables t{ws};
    Walk w(t, 1);
    w.take_slices(t, plan.size() - 1);
    if ((rc = t.open()) || (rc = put_walk(t, w, d_fasta, offs, &plan, s))) return rc;
    *out = DevWalk{t.dev<GenomeDev>(w.genomes), t.dev<Slice>(w.slices), w.n_slices};
    return KMERML_OK;
}

// Global-atomic counting: ~8 slices per SM over the genome, each of 1 to 64 tiles.
static uint64_t atomic_slice_bytes(int sm_count, uint64_t genome_bytes) {
    const uint64_t target = (uint64_t)sm_count * 8;
    return align_up(std::min<uint64_t>(std::max<uint64_t>(genome_bytes / target, TILE_BYTES), 64ull * TILE_BYTES), TILE_BYTES);
}

// The buffer and genome offsets of a multi-genome call.  counts32: every genome's windows must fit 32-bit counters.
static int check_batch(const uint8_t* d_fasta, const uint64_t* h_offsets, int n_genomes, bool counts32) {
    if (!d_fasta && h_offsets[n_genomes] > h_offsets[0]) return fail(KMERML_ERR_ARG, "d_fasta is null");
    if ((uintptr_t)d_fasta & 15) return fail(KMERML_ERR_ARG, "device pointers must be 16-byte aligned");
    for (int g = 0; g < n_genomes; g++) {
        if (h_offsets[g + 1] < h_offsets[g]) return fail(KMERML_ERR_ARG, "offsets must be non-decreasing");
        if (counts32 && h_offsets[g + 1] - h_offsets[g] >= (1ull << 32))
            return fail(KMERML_ERR_RANGE, "a genome of 4 GiB or more does not fit the 32-bit counters");
    }
    return KMERML_OK;
}

static int build_row(const int* k_list, int nk, RowSpec* row, int* kmax, int* kmin) {
    if (!k_list || nk < 1 || nk > 14) return fail(KMERML_ERR_ARG, "k_list must hold 1..14 values");
    row->nk = nk;
    unsigned long long off = 0;
    *kmax = 0;
    *kmin = 99;
    for (int i = 0; i < nk; i++) {
        int k = k_list[i];
        if (k < 1 || k > KMERML_MAX_DENSE_K)
            return fail(KMERML_ERR_ARG, "dense k must be in 1.." + std::to_string(KMERML_MAX_DENSE_K));
        for (int j = 0; j < i; j++)
            if (k_list[j] == k) return fail(KMERML_ERR_ARG, "k_list values must be distinct");
        row->k[i] = k;
        row->off[i] = off;
        off += 1ull << (2 * k);
        *kmax = std::max(*kmax, k);
        *kmin = std::min(*kmin, k);
    }
    row->off[nk] = off;
    return KMERML_OK;
}

// The dense path on device-resident bytes, using one workspace, asynchronous on `s`.
static int count_dense_core(kmerml_ctx* ctx, Workspace& ws, const uint8_t* d_fasta, const uint64_t* h_offsets,
                            int n_genomes, const int* k_list, int nk, int min_record_len, unsigned flags,
                            uint32_t* d_counts, uint64_t counts_stride, float* d_freq, uint64_t freq_stride,
                            uint64_t* d_totals, cudaStream_t s, uint64_t range_begin = 0, uint64_t range_end = 0) {
    RowSpec row;
    int kmax, kmin;
    int rc = build_row(k_list, nk, &row, &kmax, &kmin);
    if (rc) return rc;
    if (n_genomes < 0) return fail(KMERML_ERR_ARG, "n_genomes < 0");
    if (n_genomes == 0) return KMERML_OK;
    if (!h_offsets || !d_counts) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (counts_stride < row.off[nk] || (counts_stride & 3))
        return fail(KMERML_ERR_ARG, "counts_stride must be >= row length and a multiple of 4");
    if (d_freq && (freq_stride < row.off[nk] || (freq_stride & 3)))
        return fail(KMERML_ERR_ARG, "freq_stride must be >= row length and a multiple of 4");
    int min_rec = min_record_len > 0 ? min_record_len : kmax;
    if (min_rec < kmax) return fail(KMERML_ERR_ARG, "min_record_len must be >= max(k_list)");
    if (((uintptr_t)d_counts & 15) || (d_freq && ((uintptr_t)d_freq & 15)))
        return fail(KMERML_ERR_ARG, "device pointers must be 16-byte aligned");
    if ((rc = check_batch(d_fasta, h_offsets, n_genomes, true))) return rc;
    // the level that is actually counted; every lower level comes from the cascade.  k = 8 does not
    // fit the shared histogram of count_kernel<1> (256 KB), so it is counted as 9-mers through the
    // partition path (level 9 is a pass-through scratch level) instead of with global atomics
    const bool part_ok = !(flags & KMERML_FLAG_NO_PARTITION);
    // k = 8: packed 16-bit shared histogram (count8_kernel); KMERML_FLAG_K8_AS_9 counts 9-mers through
    // the partition path instead (kept for comparison)
    const int kcount = (kmax == SMEM_MAX_K + 1 && part_ok && (flags & KMERML_FLAG_K8_AS_9)) ? PART_MIN_K : kmax;
    const bool use_smem = kcount <= SMEM_MAX_K + 1;
    const bool use_part = kcount >= PART_MIN_K && kcount <= PART_MAX_K && part_ok;
    const bool canonical = (flags & KMERML_FLAG_CANONICAL) != 0;

    // ---- level map: requested levels live in the caller's row, the rest in scratch
    LevelMap lm;
    memset(&lm, 0, sizeof(lm));
    unsigned long long scratch_stride = 0;
    for (int j = kmin; j <= kcount; j++) {
        int ki = -1;
        for (int i = 0; i < nk; i++)
            if (row.k[i] == j) ki = i;
        if (ki >= 0) {
            lm.off[j] = (long long)row.off[ki];
        } else {
            lm.off[j] = -1 - (long long)scratch_stride;
            scratch_stride += 1ull << (2 * j);
        }
    }
    lm.counts = d_counts;
    lm.counts_stride = counts_stride;
    lm.scratch_slots = (use_smem || use_part) ? (uint32_t)n_genomes : 1u;
    lm.scratch_stride = scratch_stride;
    if (scratch_stride) {
        rc = ws.scratch.ensure((size_t)scratch_stride * lm.scratch_slots * 4);
        if (rc) return rc;
    }
    lm.scratch = (uint32_t*)ws.scratch.p;

    // ---- slices
    const uint64_t total_bytes = h_offsets[n_genomes] - h_offsets[0];
    const uint64_t target = (uint64_t)ctx->sm_count * 8;
    // partition path: long runs of tiles per CTA amortise its set-up (fill of the staging buffer, first load,
    // final reduction), but a small batch needs enough CTAs to fill the GPU
    // (a byte-range call -- one rank's share of a genome -- only walks the range: size the runs from it, or a rank
    // of an 8-GPU job is left with 1.3 waves of CTAs)
    uint64_t walked_bytes = total_bytes;
    if (range_end) walked_bytes = std::min(total_bytes, range_end > range_begin ? range_end - range_begin : 0);
    // Run length T (tiles per partition CTA): the longest T <= 64 for which the runs fill a whole number of waves of
    // the 2 CTAs per SM -- w waves of (2 x SMs) runs at 96 % fill, so that genome ends (partial runs) do not spill
    // into one more wave.  (Powers of two left a rank of an 8-GPU job with 5.03 waves: six rounds for 84 % use.)
    int part_tiles_per_slice = 1;
    {
        const uint64_t tiles = std::max<uint64_t>(walked_bytes / TILE_BYTES, 1);
        const uint64_t slots = (uint64_t)ctx->sm_count * 2;
        for (uint64_t w = 1;; w++) {
            const uint64_t t = (tiles * 100 + slots * w * 96 - 1) / (slots * w * 96);
            if (t <= (uint64_t)PART_MAX_TILES_PER_RUN) {
                part_tiles_per_slice = (int)std::max<uint64_t>(t, 1);
                break;
            }
        }
    }
    if (const char* e = getenv("KMERML_TILES_PER_RUN")) {      // profiling hook: the run length of a big batch on a small one
        const int v = atoi(e);
        if (v >= 1 && v <= PART_MAX_TILES_PER_RUN) part_tiles_per_slice = v;
    }
    std::vector<uint64_t> slice_bytes(n_genomes);
    for (int g = 0; g < n_genomes; g++) {
        if (use_part)
            slice_bytes[g] = (uint64_t)TILE_BYTES * part_tiles_per_slice;   // a CTA walks a run of consecutive tiles
        else if (use_smem)
            slice_bytes[g] = (uint64_t)n_genomes >= target ? 1ull << 40      // a genome per CTA
                             : align_up(std::max<uint64_t>(total_bytes / target, 4ull * TILE_BYTES), TILE_BYTES);
        else
            slice_bytes[g] = atomic_slice_bytes(ctx->sm_count, h_offsets[g + 1] - h_offsets[g]);
    }
    std::vector<Slice> plan;
    std::vector<uint32_t> first_slice;
    rc = plan_slices(h_offsets, n_genomes, slice_bytes.data(), TILE_BYTES, range_begin, range_end, plan, first_slice);
    if (rc) return rc;
    const uint64_t n_slices = first_slice[n_genomes];
    // ---- tables: the walk | partition path: genome -> (first run, runs)
    Tables t{ws};
    Walk walk(t, n_genomes);
    walk.take_slices(t, n_slices);
    const size_t at_gruns = t.take((size_t)n_genomes * 8);
    if ((rc = t.open())) return rc;
    const GenomeDev* d_genomes = t.dev<GenomeDev>(walk.genomes);
    GenomeStats* d_stats = t.dev<GenomeStats>(walk.stats);
    const Slice* d_slices = t.dev<Slice>(walk.slices);
    // partition path: genomes are processed in groups whose payload workspace is bounded; a slice is a run
    // (the tiles one partition CTA walks), and a run's regions take tiles_per_run * 64 KB of payload
    std::vector<int> group_end;                              // exclusive genome index per group
    const uint64_t run_payload_bytes = (uint64_t)part_tiles_per_slice * PART_STAGE_ENTRIES * 2;
    if (use_part) {
        uint32_t* h_gruns = t.fill<uint32_t>(at_gruns, (size_t)n_genomes * 8);
        const uint64_t max_runs = std::max<uint64_t>(ctx->max_group_payload / run_payload_bytes, 1);
        uint64_t in_group = 0;
        uint32_t group_run0 = 0;
        for (int g = 0; g < n_genomes; g++) {
            const uint64_t nr = first_slice[g + 1] - first_slice[g];
            if (in_group && in_group + nr > max_runs) {
                group_end.push_back(g);
                in_group = 0;
                group_run0 = first_slice[g];
            }
            h_gruns[2 * g] = first_slice[g] - group_run0;    // run numbers are relative to the group's first run
            h_gruns[2 * g + 1] = (uint32_t)nr;
            in_group += nr;
        }
        group_end.push_back(n_genomes);
    }
    {
        Prof pr(ctx, s, 3, 4);      // prologue + the three slice-table kernels
        rc = put_walk(t, walk, d_fasta, h_offsets, &plan, s);
    }
    if (rc) return rc;
    const int n_cascade = cascade_launches(kcount, kmin);

    const size_t row_bytes = (size_t)row.off[nk] * 4;
    if (use_part) {
        const int k_stop = std::max(kcount - PART_LOW_BASES, kmin);
        uint64_t max_group_runs = 0, max_group_bytes = 0, max_group_genomes = 0;
        for (size_t gi = 0, g0 = 0; gi < group_end.size(); g0 = group_end[gi], gi++) {
            max_group_runs = std::max<uint64_t>(max_group_runs, first_slice[group_end[gi]] - first_slice[g0]);
            max_group_bytes = std::max<uint64_t>(max_group_bytes, h_offsets[group_end[gi]] - h_offsets[g0]);
            max_group_genomes = std::max<uint64_t>(max_group_genomes, group_end[gi] - g0);
        }
        const int nb = 1 << (2 * (kcount - PART_LOW_BASES));
        // workspace: payload regions [run][bucket][cap sectors] | sectors written per (run, bucket) |
        // overflow lists (one entry per FASTA byte at most) | ...
        const size_t payload_bytes = align_up((size_t)max_group_runs * run_payload_bytes, 256);
        const size_t nsec_bytes = align_up((size_t)max_group_runs * nb * 2, 256);
        const size_t ov_bytes = align_up((size_t)max_group_bytes * 4 + 64, 256);
        // ... | run-end tail lists (one entry per 64 FASTA bytes + 1024 per genome) | counters (overflow, tails)
        const size_t ovc_bytes = align_up((size_t)n_genomes * 8 + 8, 256);
        const size_t tl_bytes = align_up((size_t)((max_group_bytes >> 6) + 1024 * (max_group_genomes + 1)) * 8, 256);
        rc = ws.part.ensure(payload_bytes + nsec_bytes + ov_bytes + tl_bytes + ovc_bytes);
        if (rc) return rc;
        uint8_t* pw = (uint8_t*)ws.part.p;
        void* d_payload = pw;
        uint16_t* d_nsec = (uint16_t*)(pw + payload_bytes);
        uint32_t* d_overflow = (uint32_t*)(pw + payload_bytes + nsec_bytes);
        unsigned long long* d_tail_list = (unsigned long long*)(pw + payload_bytes + nsec_bytes + ov_bytes);
        unsigned int* d_ov_counts = (unsigned int*)(pw + payload_bytes + nsec_bytes + ov_bytes + tl_bytes);
        unsigned int* d_tail_counts = d_ov_counts + n_genomes;
        unsigned int* d_tail_any = d_tail_counts + n_genomes;
        KM_CUDA(cudaMemsetAsync(d_ov_counts, 0, (size_t)n_genomes * 8 + 8, s));
        // the bucket kernel stores every row from level k_stop upwards in full; only the few small
        // levels below it collect run-end tails directly and must start from zero
        for (int i = 0; i < nk; i++)
            if (row.k[i] < k_stop)
                KM_CUDA(cudaMemset2DAsync(d_counts + row.off[i], (size_t)counts_stride * 4, 0,
                                          (size_t)(1ull << (2 * row.k[i])) * 4, (size_t)n_genomes, s));
        if (scratch_stride && k_stop > kmin)
            KM_CUDA(cudaMemsetAsync(lm.scratch, 0, (size_t)scratch_stride * n_genomes * 4, s));
        int g0 = 0;
        for (size_t gi = 0; gi < group_end.size(); gi++) {
            const int g1 = group_end[gi], ng = g1 - g0;
            const int nt = (int)(first_slice[g1] - first_slice[g0]);
            const uint64_t batch_lo = h_offsets[g0];
            {
                Prof pr(ctx, s, 4, nt > 0 ? 1 : 0);
                rc = launch_partition(d_fasta, d_genomes, d_slices + first_slice[g0], nt, part_tiles_per_slice, kcount,
                                      kmin, min_rec, lm, d_stats, d_payload, d_nsec, d_overflow, d_ov_counts, batch_lo,
                                      d_tail_list, d_tail_counts, d_tail_any, (uint32_t)g0, s);
            }
            if (rc) return rc;
            {
                Prof pr(ctx, s, 5, 1);
                rc = launch_bucket(lm, row, kcount, kmin, t.dev<uint32_t>(at_gruns), part_tiles_per_slice, d_payload, d_nsec, d_stats,
                                   canonical ? nullptr : d_freq, freq_stride, d_totals, (uint32_t)g0, ng, s);
            }
            if (rc) return rc;
            if (kcount > kmin) {
                Prof pr(ctx, s, 3, canonical || !d_freq ? 2 : 4);
                rc = launch_tails(d_fasta, lm, row, kcount, kmin, min_rec, d_genomes, d_slices + first_slice[g0], nt,
                                  d_tail_list, d_tail_counts, d_tail_any, batch_lo, d_stats, canonical ? nullptr : d_freq, freq_stride,
                                  (uint32_t)g0, ng, s);
                if (rc) return rc;
            }
            for (int h0 = g0; h0 < g1; h0 += 32768) {
                const int nh = std::min(32768, g1 - h0);
                {
                    Prof pr(ctx, s, 3, canonical || !d_freq ? 1 : 2);
                    rc = launch_overflow(lm, row, kcount, kmin, d_genomes, d_overflow, d_ov_counts, batch_lo, d_stats,
                                         canonical ? nullptr : d_freq, freq_stride, (uint32_t)h0, nh, s);
                    if (rc) return rc;
                }
                if (k_stop > kmin) {
                    Prof pr(ctx, s, 1, cascade_launches(k_stop, kmin));
                    rc = launch_cascade(lm, k_stop, kmin, (uint32_t)h0, nh, s);
                    if (rc) return rc;
                }
                Prof pr(ctx, s, 2, canonical ? finalize_launches(row, true) : 1);
                if (canonical)
                    rc = launch_finalize(lm, row, kcount, true, d_stats, d_freq, freq_stride, d_totals, (uint32_t)h0, nh, s);
                else
                    rc = launch_finalize_low(lm, row, kcount, k_stop, d_stats, d_freq, freq_stride, (uint32_t)h0, nh, s);
                if (rc) return rc;
            }
            g0 = g1;
        }
    } else if (use_smem) {
        KM_CUDA(cudaMemset2DAsync(d_counts, (size_t)counts_stride * 4, 0, row_bytes, (size_t)n_genomes, s));
        if (scratch_stride) KM_CUDA(cudaMemsetAsync(lm.scratch, 0, (size_t)scratch_stride * n_genomes * 4, s));
        {
            Prof pr(ctx, s, 0, 1);
            rc = launch_count(d_fasta, d_genomes, d_slices, (int)n_slices, kcount, kmin, min_rec, true, lm, d_stats, s);
        }
        if (rc) return rc;
        for (int g0 = 0; g0 < n_genomes; g0 += 32768) {
            int ng = std::min(32768, n_genomes - g0);
            {
                Prof pr(ctx, s, 1, n_cascade);
                rc = launch_cascade(lm, kcount, kmin, (uint32_t)g0, ng, s);
            }
            if (rc) return rc;
            {
                Prof pr(ctx, s, 2, finalize_launches(row, canonical));
                rc = launch_finalize(lm, row, kcount, canonical, d_stats, d_freq, freq_stride, d_totals, (uint32_t)g0, ng, s);
            }
            if (rc) return rc;
        }
    } else {
        // one genome at a time so that its 4^k row stays resident in the 126 MB L2
        for (int g = 0; g < n_genomes; g++) {
            KM_CUDA(cudaMemsetAsync(d_counts + (size_t)g * counts_stride, 0, row_bytes, s));
            if (scratch_stride) KM_CUDA(cudaMemsetAsync(lm.scratch, 0, (size_t)scratch_stride * 4, s));
            int ns = (int)(first_slice[g + 1] - first_slice[g]);
            {
                Prof pr(ctx, s, 0, ns > 0 ? 1 : 0);
                rc = launch_count(d_fasta, d_genomes, d_slices + first_slice[g], ns, kcount, kmin, min_rec, false, lm, d_stats, s);
            }
            if (rc) return rc;
            {
                Prof pr(ctx, s, 1, n_cascade);
                rc = launch_cascade(lm, kcount, kmin, (uint32_t)g, 1, s);
            }
            if (rc) return rc;
            {
                Prof pr(ctx, s, 2, finalize_launches(row, canonical));
                rc = launch_finalize(lm, row, kcount, canonical, d_stats, d_freq, freq_stride, d_totals, (uint32_t)g, 1, s);
            }
            if (rc) return rc;
        }
    }
    return KMERML_OK;
}

// A batch whose genome g occupies [starts[g], starts[g] + sizes[g]) of the buffer (starts are 256-byte aligned, so
// there may be gaps): the core takes back-to-back offsets, and bytes between a genome's end and the next start
// would be read as FASTA text, so the gaps must hold no text: they are filled with line feeds here.
static int count_dense_group(kmerml_ctx* ctx, Workspace& ws, const uint8_t* d_fasta, const uint64_t* starts,
                             const uint64_t* sizes, int n, const int* k_list, int nk, int min_record_len, unsigned flags,
                             uint32_t* d_counts, uint64_t counts_stride, float* d_freq, uint64_t freq_stride,
                             uint64_t* d_totals, cudaStream_t s) {
    for (int g = 0; g < n; g++) {
        const uint64_t end = starts[g] + sizes[g];
        if (starts[g + 1] > end)
            KM_CUDA(cudaMemsetAsync(const_cast<uint8_t*>(d_fasta) + end, '\n', (size_t)(starts[g + 1] - end), s));
    }
    return count_dense_core(ctx, ws, d_fasta, starts, n, k_list, nk, min_record_len, flags, d_counts, counts_stride, d_freq,
                            freq_stride, d_totals, s);
}

}  // namespace km

using namespace km;

extern "C" {

int kmerml_version(void) { return 100; }

const char* kmerml_last_error(void) { return g_err.c_str(); }

int kmerml_ctx_create(int device, kmerml_ctx** out) {
    if (!out) return fail(KMERML_ERR_ARG, "out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        (void)cudaGetLastError();
        return fail(KMERML_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= n) return fail(KMERML_ERR_ARG, "device index out of range");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop;
    KM_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(KMERML_ERR_CUDA, std::string("built for sm_100a (B200); device is ") + prop.name);
    kmerml_ctx* ctx = new (std::nothrow) kmerml_ctx();
    if (!ctx) return fail(KMERML_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (const char* hs = getenv("KMERML_HOST_SLOTS")) {                // pipeline depth of the host-buffer call
        const int v = atoi(hs);
        if (v >= 1 && v <= 8) ctx->host_slots = v;
    }
    if (const char* mb = getenv("KMERML_GROUP_PAYLOAD_MB")) {      // smaller groups: less workspace (and a test hook)
        const long long v = atoll(mb);
        if (v > 0) ctx->max_group_payload = (uint64_t)v << 20;
    }
    int rc = dense_setup_attributes();
    if (rc) { delete ctx; return rc; }
    *out = ctx;
    return KMERML_OK;
}

int kmerml_ctx_destroy(kmerml_ctx* ctx) {
    if (!ctx) return KMERML_OK;
    DeviceGuard guard(ctx->device);
    cudaDeviceSynchronize();
    for (auto& w : ctx->ws) w.release();
    ctx->fmh_kept.release();
    ctx->fmh_index.release();
    ctx->fmh_abund.release();
    if (ctx->order_ev) cudaEventDestroy(ctx->order_ev);
    if (ctx->host_pool) host_pool_destroy(ctx->host_pool);
    for (auto& r : ctx->recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : ctx->pool) cudaEventDestroy(e);
    delete ctx;
    return KMERML_OK;
}

int kmerml_ctx_sm_count(const kmerml_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

int kmerml_ctx_set_host_threads(kmerml_ctx* ctx, int n_threads) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (n_threads < 1 || n_threads > 256) return fail(KMERML_ERR_ARG, "n_threads must be in 1..256");
    if (ctx->host_pool && host_pool_size(ctx->host_pool) == n_threads) return KMERML_OK;
    if (ctx->host_pool) host_pool_destroy(ctx->host_pool);
    ctx->host_pool = host_pool_create(n_threads);
    if (!ctx->host_pool) return fail(KMERML_ERR_NOMEM, "could not start the host thread pool");
    return KMERML_OK;
}

int kmerml_profile_enable(kmerml_ctx* ctx, int on) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    ctx->profiling = on != 0;
    return KMERML_OK;
}

int kmerml_profile_read(kmerml_ctx* ctx, kmerml_profile* out, int reset) {
    if (!ctx || !out) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    for (auto& r : ctx->recs) {
        KM_CUDA(cudaEventSynchronize(r.b));
        float ms = 0;
        KM_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
        ctx->ms[r.kind] += ms;
        ctx->pool.push_back(r.a);
        ctx->pool.push_back(r.b);
    }
    ctx->recs.clear();
    out->launches = ctx->launches;
    out->count_launches = ctx->count_launches;
    out->ms_count = ctx->ms[0];
    out->ms_cascade = ctx->ms[1];
    out->ms_finalize = ctx->ms[2];
    out->ms_other = ctx->ms[3];
    out->ms_partition = ctx->ms[4];
    out->ms_bucket = ctx->ms[5];
    if (reset) {
        ctx->launches = ctx->count_launches = 0;
        for (double& m : ctx->ms) m = 0;
    }
    return KMERML_OK;
}

uint64_t kmerml_row_len(const int* k_list, int nk) {
    uint64_t n = 0;
    for (int i = 0; k_list && i < nk; i++)
        if (k_list[i] >= 0 && k_list[i] <= 31) n += 1ull << (2 * k_list[i]);
    return n;
}

int kmerml_count_dense_batch(kmerml_ctx* ctx, const uint8_t* d_fasta, const uint64_t* h_offsets, int n_genomes,
                             const int* k_list, int nk, int min_record_len, unsigned flags, uint32_t* d_counts,
                             uint64_t counts_stride, float* d_freq, uint64_t freq_stride, uint64_t* d_totals,
                             void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return count_dense_core(ctx, ctx->ws[0], d_fasta, h_offsets, n_genomes, k_list, nk, min_record_len, flags,
                            d_counts, counts_stride, d_freq, freq_stride, d_totals, (cudaStream_t)stream);
}

int kmerml_count_dense_range(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin,
                             uint64_t range_end, const int* k_list, int nk, int min_record_len, unsigned flags,
                             uint32_t* d_counts, uint64_t* d_totals, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (range_begin % TILE_BYTES) return fail(KMERML_ERR_ARG, "range_begin must be a multiple of 16384");
    if (range_end > nbytes) range_end = nbytes;
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    uint64_t offs[2] = {0, nbytes};
    RowSpec row;
    int kmax, kmin;
    int rc = build_row(k_list, nk, &row, &kmax, &kmin);
    if (rc) return rc;
    if (range_begin >= range_end) {                       // empty range: an all-zero contribution
        KM_CUDA(cudaMemsetAsync(d_counts, 0, (size_t)row.off[nk] * 4, (cudaStream_t)stream));
        if (d_totals) KM_CUDA(cudaMemsetAsync(d_totals, 0, (size_t)nk * 8, (cudaStream_t)stream));
        return KMERML_OK;
    }
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return count_dense_core(ctx, ctx->ws[0], d_fasta, offs, 1, k_list, nk, min_record_len, flags, d_counts,
                            align_up((size_t)row.off[nk], 4), nullptr, 0, d_totals, (cudaStream_t)stream, range_begin,
                            range_end);
}

namespace {

constexpr int NARROW_MIN_K = 10;                 // levels that cross the bus as one byte (or one nibble) per bin
constexpr uint32_t NARROW_EXC_CAP = 32768;       // exception list entries (bin, count) per genome
constexpr uint32_t WIRE_MAGIC = 0x32574D4Bu;     // "KMW2": header word 0 of a wire row; word 1 = nibble mask over k_list
constexpr size_t WIRE_HEADER = 16;
constexpr size_t NARROW_CHUNK = 1u << 20;        // bins one host task widens
// Measured (1 x B200, C2): the call is bound by the box's host memory system (~60 GB/s of DMA traffic in either
// direction), not by launches: 8 genomes per slot gave the same 86 ms per step for the compact result and made the
// uint32 variant slower (a group's rows can only be widened once its last byte has arrived), so a slot holds one.
constexpr int HOST_GROUP_MAX = 1;                // genomes one pipeline slot holds (one batch of kernels) ...
constexpr uint64_t HOST_GROUP_BYTES = 192ull << 20;   // ... and their FASTA bytes, at most

// wire row of one genome:
//   [header 16 B | narrow block | exception count (16 B) | exception list | small levels (uint32)]
// nibble_mask bit i: level i of k_list is packed two bins per byte
struct WireLayout {
    km::NarrowSpec spec;
    uint32_t nibble_mask;
    size_t narrow_off, exc_off, small_off, bytes;
};

WireLayout wire_layout(const km::RowSpec& row, bool narrow_big_levels, uint32_t nibble_mask) {
    WireLayout L;
    memset(&L, 0, sizeof(L));
    km::NarrowSpec& sp = L.spec;
    unsigned long long small = 0;
    for (int i = 0; i < row.nk; i++) {
        const unsigned long long n = 1ull << (2 * row.k[i]);
        if (narrow_big_levels && row.k[i] >= NARROW_MIN_K) {
            const bool nib = (nibble_mask >> i) & 1u;
            if (nib) L.nibble_mask |= 1u << i;
            sp.src_off[sp.n] = row.off[i];
            sp.dst_off[sp.n] = sp.total;
            sp.nibble[sp.n] = nib ? 1 : 0;
            sp.total += nib ? n / 2 : n;
            sp.n++;
        } else {
            sp.small_src[sp.n_small] = row.off[i];
            sp.small_dst[sp.n_small] = small;
            small += n;
            sp.n_small++;
        }
    }
    sp.dst_off[sp.n] = sp.total;
    sp.small_dst[sp.n_small] = small;
    sp.small_total = small;
    L.narrow_off = WIRE_HEADER;
    L.exc_off = L.narrow_off + (size_t)sp.total;
    L.small_off = L.exc_off + 16 + (size_t)NARROW_EXC_CAP * 8;
    L.bytes = (L.small_off + (size_t)small * 4 + 15) / 16 * 16;
    return L;
}

// Which levels of a genome of `fasta_bytes` bytes go as nibbles: those with a mean count <= 5 (Poisson(5) reaches 15
// with probability 7e-5: a few hundred exceptions per 4^12 bins); repeats beyond that land in the exception list, and
// a list that overflows sends the genome again in full.
uint32_t nibble_mask_for(const km::RowSpec& row, uint64_t fasta_bytes) {
    uint32_t m = 0;
    for (int i = 0; i < row.nk; i++)
        if (row.k[i] >= NARROW_MIN_K && fasta_bytes <= 5ull << (2 * row.k[i])) m |= 1u << i;
    return m;
}

struct HostSlot {                                // hand-over between the stream callback, the pool and the caller
    std::mutex m;
    std::condition_variable cv;
    bool busy = false;                           // a group's expansion is outstanding
    bool overflow[HOST_GROUP_MAX] = {};          // exception list overflowed: the caller copies that row in full
    std::atomic<int> remaining{0};
    // the group in the slot
    int n = 0;
    const uint8_t* wire_host = nullptr;          // n wire rows, wire_stride bytes apart
    size_t wire_stride = 0;
    uint32_t* row[HOST_GROUP_MAX] = {};          // the caller's uint32 rows
    WireLayout lay;
    km::HostPool* pool = nullptr;
};

void slot_finish(HostSlot* sl) {                 // last task of a group: exceptions, then the slot is free
    bool over[HOST_GROUP_MAX] = {};
    for (int g = 0; g < sl->n; g++) {
        const uint8_t* tail = sl->wire_host + (size_t)g * sl->wire_stride + sl->lay.exc_off;
        uint32_t n_exc;
        memcpy(&n_exc, tail, 4);
        over[g] = n_exc > NARROW_EXC_CAP;
        if (!over[g]) {
            const uint32_t* e = reinterpret_cast<const uint32_t*>(tail + 16);
            for (uint32_t i = 0; i < n_exc; i++) sl->row[g][e[2 * i]] = e[2 * i + 1];
        }
    }
    {
        std::lock_guard<std::mutex> lk(sl->m);
        for (int g = 0; g < sl->n; g++) sl->overflow[g] = over[g];
        sl->busy = false;
    }
    sl->cv.notify_all();
}

void CUDART_CB slot_arrived(void* p) {           // stream callback: the group's wire rows are in host memory
    HostSlot* sl = static_cast<HostSlot*>(p);
    const km::NarrowSpec& sp = sl->lay.spec;
    int per_genome = sp.n_small ? 1 : 0;
    for (int i = 0; i < sp.n; i++) per_genome += (int)((sp.dst_off[i + 1] - sp.dst_off[i] + NARROW_CHUNK - 1) / NARROW_CHUNK);
    if (!per_genome || !sl->n) { slot_finish(sl); return; }
    sl->remaining.store(per_genome * sl->n);
    for (int g = 0; g < sl->n; g++) {
        const uint8_t* wire = sl->wire_host + (size_t)g * sl->wire_stride;
        uint32_t* row = sl->row[g];
        if (sp.n_small) {
            const km::NarrowSpec* spp = &sl->lay.spec;
            const uint8_t* small = wire + sl->lay.small_off;
            km::host_pool_submit(sl->pool, [sl, spp, small, row] {
                for (int i = 0; i < spp->n_small; i++)
                    memcpy(row + spp->small_src[i], small + spp->small_dst[i] * 4,
                           (size_t)(spp->small_dst[i + 1] - spp->small_dst[i]) * 4);
                if (sl->remaining.fetch_sub(1) == 1) slot_finish(sl);
            });
        }
        for (int i = 0; i < sp.n; i++) {
            const size_t len = (size_t)(sp.dst_off[i + 1] - sp.dst_off[i]);
            const bool nib = sp.nibble[i] != 0;
            for (size_t c = 0; c < len; c += NARROW_CHUNK) {
                const uint8_t* src = wire + sl->lay.narrow_off + sp.dst_off[i] + c;
                uint32_t* dst = row + sp.src_off[i] + (nib ? 2 * c : c);
                const size_t n = std::min(NARROW_CHUNK, len - c);
                km::host_pool_submit(sl->pool, [sl, src, dst, n, nib] {
                    if (nib) km::widen_u4_to_u32(src, dst, n);
                    else km::widen_u8_to_u32(src, dst, n);
                    if (sl->remaining.fetch_sub(1) == 1) slot_finish(sl);
                });
            }
        }
    }
}

}  // namespace

// compact_rows != nullptr: the wire rows are delivered as they crossed the bus (kmerml_count_dense_host_compact),
// one row of `compact_stride` bytes per genome.  Genomes travel in groups of up to HOST_GROUP_MAX per pipeline slot
// (three slots): one H2D copy per genome, ONE batch of counting kernels and one narrowing kernel per group, one D2H
// copy per genome.
static int count_dense_host_impl(kmerml_ctx* ctx, const uint8_t* const* h_fasta, const uint64_t* h_sizes, int n_genomes,
                                 const int* k_list, int nk, int min_record_len, unsigned flags, uint32_t* h_counts,
                                 uint64_t counts_stride, float* freq, uint64_t freq_stride, uint64_t* h_totals,
                                 uint8_t* compact_rows, uint64_t compact_stride) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (n_genomes < 0) return fail(KMERML_ERR_ARG, "n_genomes < 0");
    if (n_genomes == 0) return KMERML_OK;
    const bool compact = compact_rows != nullptr;
    if (!h_fasta || !h_sizes || (!h_counts && !compact)) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    // slot 0 shares ws[0] with the device-resident calls: let what the last of them launched finish first
    // (this call runs on its own streams and returns synchronised)
    if (ctx->last_stream_valid) {
        if (cudaStreamSynchronize(ctx->last_stream) != cudaSuccess) {
            (void)cudaGetLastError();
            KM_CUDA(cudaDeviceSynchronize());
        }
        ctx->last_stream_valid = false;
    }
    RowSpec row;
    int kmax, kmin;
    int rc = build_row(k_list, nk, &row, &kmax, &kmin);
    if (rc) return rc;
    const bool freq_dev = freq && (flags & KMERML_FLAG_FREQ_ON_DEVICE);
    const size_t row_len = (size_t)row.off[nk];
    const size_t row_stride = align_up(row_len, 4);
    if (!compact && counts_stride < row_len) return fail(KMERML_ERR_ARG, "counts_stride must be >= row length");
    if (freq_dev && (((uintptr_t)freq & 15) || (freq_stride & 3) || freq_stride < row_len))
        return fail(KMERML_ERR_ARG, "device freq buffer must be 16-byte aligned with a stride multiple of 4");
    // the levels k >= 10 cross the bus as bytes + exceptions (hostpipe.cu), the small ones as they are
    const bool wire = compact || !(flags & KMERML_FLAG_WIDE_D2H);
    const WireLayout lay_max = wire_layout(row, true, 0);           // all levels as bytes: the largest row
    if (compact && compact_stride < lay_max.bytes)
        return fail(KMERML_ERR_ARG, "compact row stride smaller than kmerml_compact_row_bytes");
    if (wire && !compact && !ctx->host_pool) {
        int n_thr = 0;
        if (const char* e = getenv("KMERML_HOST_THREADS")) n_thr = atoi(e);
        if (n_thr <= 0) n_thr = (int)std::min(16u, std::max(2u, std::thread::hardware_concurrency() / 2));
        ctx->host_pool = host_pool_create(n_thr);
        if (!ctx->host_pool) return fail(KMERML_ERR_NOMEM, "could not start the host thread pool");
    }
    // groups of consecutive genomes
    std::vector<int> group_begin;
    {
        uint64_t bytes = 0;
        int cnt = 0;
        for (int g = 0; g < n_genomes; g++) {
            if (h_sizes[g] >= (1ull << 32)) return fail(KMERML_ERR_RANGE, "a genome of 4 GiB or more does not fit the 32-bit counters");
            if (cnt == 0 || cnt >= HOST_GROUP_MAX || bytes + h_sizes[g] > HOST_GROUP_BYTES) {
                group_begin.push_back(g);
                bytes = 0;
                cnt = 0;
            }
            bytes += h_sizes[g];
            cnt++;
        }
        group_begin.push_back(n_genomes);
    }
    const int n_groups = (int)group_begin.size() - 1;
    uint64_t max_group_bytes = 0;
    int max_group = 0;
    for (int gi = 0; gi < n_groups; gi++) {
        uint64_t b = 0;
        for (int g = group_begin[gi]; g < group_begin[gi + 1]; g++) b += align_up((size_t)h_sizes[g], 256);
        max_group_bytes = std::max(max_group_bytes, b);
        max_group = std::max(max_group, group_begin[gi + 1] - group_begin[gi]);
    }
    const int n_slots = std::min(ctx->host_slots, n_groups);
    std::unique_ptr<HostSlot[]> slots(new (std::nothrow) HostSlot[8]);
    if (!slots) return fail(KMERML_ERR_NOMEM, "out of host memory");
    for (int i = 0; i < n_slots; i++) {
        Workspace& w = ctx->ws[i];
        if (!w.stream) KM_CUDA(cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
        if ((rc = w.fasta.ensure(align_up((size_t)max_group_bytes + 64, 256)))) return rc;
        if ((rc = w.counts.ensure((size_t)max_group * row_stride * 4))) return rc;
        if (freq && !freq_dev && (rc = w.freq.ensure((size_t)max_group * row_stride * 4))) return rc;
        if ((rc = w.totals.ensure((size_t)max_group * nk * 8))) return rc;
        if (wire) {
            if ((rc = w.wire.ensure((size_t)max_group * lay_max.bytes))) return rc;
            if (!compact && (rc = w.wire_host.ensure((size_t)max_group * lay_max.bytes))) return rc;
        }
    }
    // every exit below first waits for the host tasks that still reference `slots`
    auto wait_slot = [&](int si, int group) -> int {
        HostSlot& sl = slots[si];
        std::unique_lock<std::mutex> lk(sl.m);
        sl.cv.wait(lk, [&] { return !sl.busy; });
        for (int j = 0; j < sl.n; j++) {
            if (!sl.overflow[j]) continue;       // more than NARROW_EXC_CAP bins >= 255: that row in full
            sl.overflow[j] = false;
            KM_CUDA(cudaMemcpy(h_counts + (size_t)(group_begin[group] + j) * counts_stride,
                               (uint32_t*)ctx->ws[si].counts.p + (size_t)j * row_stride, row_len * 4, cudaMemcpyDeviceToHost));
        }
        return KMERML_OK;
    };
    auto drain = [&]() {
        for (int i = 0; i < n_slots; i++) cudaStreamSynchronize(ctx->ws[i].stream);
        for (int i = 0; i < n_slots; i++) {
            std::unique_lock<std::mutex> lk(slots[i].m);
            slots[i].cv.wait(lk, [&] { return !slots[i].busy; });
        }
    };
#define KM_HOST_TRY(expr)                                                     \
    do {                                                                      \
        cudaError_t e__ = (expr);                                             \
        if (e__ != cudaSuccess) { drain(); return cuda_fail(e__, #expr); }    \
    } while (0)
    for (int gi = 0; gi < n_groups; gi++) {
        const int si = gi % n_slots, g0 = group_begin[gi], ng = group_begin[gi + 1] - g0;
        Workspace& w = ctx->ws[si];
        cudaStream_t s = w.stream;
        if (wire && !compact && gi >= n_slots && (rc = wait_slot(si, gi - n_slots))) { drain(); return rc; }
        std::vector<uint64_t> offs(ng + 1, 0);
        for (int j = 0; j < ng; j++) {
            if (h_sizes[g0 + j])
                KM_HOST_TRY(cudaMemcpyAsync((uint8_t*)w.fasta.p + offs[j], h_fasta[g0 + j], (size_t)h_sizes[g0 + j],
                                            cudaMemcpyHostToDevice, s));
            offs[j + 1] = offs[j] + align_up((size_t)h_sizes[g0 + j], 256);
        }
        // (genomes start at 256-byte multiples of the slot's buffer; count_dense_group blanks the gaps)
        float* d_f = !freq ? nullptr : (freq_dev ? freq + (size_t)g0 * freq_stride : (float*)w.freq.p);
        rc = count_dense_group(ctx, w, (const uint8_t*)w.fasta.p, offs.data(), h_sizes + g0, ng, k_list, nk, min_record_len,
                               flags & ~(KMERML_FLAG_FREQ_ON_DEVICE | KMERML_FLAG_WIDE_D2H | KMERML_FLAG_NO_NIBBLES), (uint32_t*)w.counts.p, row_stride,
                               d_f, freq_dev ? freq_stride : row_stride, (uint64_t*)w.totals.p, s);
        if (rc) { drain(); return rc; }
        if (!wire) {
            for (int j = 0; j < ng; j++)
                KM_HOST_TRY(cudaMemcpyAsync(h_counts + (size_t)(g0 + j) * counts_stride, (uint32_t*)w.counts.p + (size_t)j * row_stride,
                                            row_len * 4, cudaMemcpyDeviceToHost, s));
        } else {
            // the group's wire layout: a level goes as nibbles when every genome of the group is small enough
            uint32_t mask = ~0u;
            for (int j = 0; j < ng; j++) mask &= nibble_mask_for(row, h_sizes[g0 + j]);
            if (flags & KMERML_FLAG_NO_NIBBLES) mask = 0;
            const WireLayout lay = wire_layout(row, true, mask);
            uint8_t* dw = (uint8_t*)w.wire.p;
            rc = launch_narrow_levels((const uint32_t*)w.counts.p, row_stride, ng, lay.spec, dw, lay_max.bytes, lay.narrow_off,
                                      lay.exc_off, lay.small_off, NARROW_EXC_CAP, WIRE_MAGIC, lay.nibble_mask, s);
            if (rc) { drain(); return rc; }
            ctx->launches += 2;
            if (compact) {
                for (int j = 0; j < ng; j++)
                    KM_HOST_TRY(cudaMemcpyAsync(compact_rows + (size_t)(g0 + j) * compact_stride, dw + (size_t)j * lay_max.bytes,
                                                lay.bytes, cudaMemcpyDeviceToHost, s));
            } else {
                for (int j = 0; j < ng; j++)
                    KM_HOST_TRY(cudaMemcpyAsync((uint8_t*)w.wire_host.p + (size_t)j * lay_max.bytes, dw + (size_t)j * lay_max.bytes,
                                                lay.bytes, cudaMemcpyDeviceToHost, s));
                HostSlot& sl = slots[si];
                {
                    std::lock_guard<std::mutex> lk(sl.m);
                    sl.busy = true;
                    for (bool& o : sl.overflow) o = false;
                }
                sl.n = ng;
                sl.wire_host = (const uint8_t*)w.wire_host.p;
                sl.wire_stride = lay_max.bytes;
                for (int j = 0; j < ng; j++) sl.row[j] = h_counts + (size_t)(g0 + j) * counts_stride;
                sl.lay = lay;
                sl.pool = ctx->host_pool;
                cudaError_t e = cudaLaunchHostFunc(s, slot_arrived, &sl);
                if (e != cudaSuccess) {
                    {
                        std::lock_guard<std::mutex> lk(sl.m);
                        sl.busy = false;
                    }
                    drain();
                    return cuda_fail(e, "cudaLaunchHostFunc");
                }
            }
        }
        if (freq && !freq_dev)
            for (int j = 0; j < ng; j++)
                KM_HOST_TRY(cudaMemcpyAsync(freq + (size_t)(g0 + j) * freq_stride, (float*)w.freq.p + (size_t)j * row_stride,
                                            row_len * 4, cudaMemcpyDeviceToHost, s));
        if (h_totals)
            KM_HOST_TRY(cudaMemcpyAsync(h_totals + (size_t)g0 * nk, w.totals.p, (size_t)ng * nk * 8, cudaMemcpyDeviceToHost, s));
    }
#undef KM_HOST_TRY
    for (int i = 0; i < n_slots; i++) KM_CUDA(cudaStreamSynchronize(ctx->ws[i].stream));
    if (wire && !compact)
        for (int gi = std::max(0, n_groups - n_slots); gi < n_groups; gi++)
            if ((rc = wait_slot(gi % n_slots, gi))) { drain(); return rc; }
    return KMERML_OK;
}

int kmerml_count_dense_host(kmerml_ctx* ctx, const uint8_t* const* h_fasta, const uint64_t* h_sizes, int n_genomes,
                            const int* k_list, int nk, int min_record_len, unsigned flags, uint32_t* h_counts,
                            uint64_t counts_stride, float* freq, uint64_t freq_stride, uint64_t* h_totals) {
    return count_dense_host_impl(ctx, h_fasta, h_sizes, n_genomes, k_list, nk, min_record_len, flags, h_counts,
                                 counts_stride, freq, freq_stride, h_totals, nullptr, 0);
}

uint64_t kmerml_compact_row_bytes(const int* k_list, int nk) {
    RowSpec row;
    int kmax, kmin;
    if (build_row(k_list, nk, &row, &kmax, &kmin)) return 0;
    return wire_layout(row, true, 0).bytes;
}

int kmerml_count_dense_host_compact(kmerml_ctx* ctx, const uint8_t* const* h_fasta, const uint64_t* h_sizes,
                                    int n_genomes, const int* k_list, int nk, int min_record_len, unsigned flags,
                                    uint8_t* h_rows, uint64_t row_stride_bytes, float* freq, uint64_t freq_stride,
                                    uint64_t* h_totals) {
    if (!h_rows) return fail(KMERML_ERR_ARG, "h_rows is null");
    if (row_stride_bytes & 15) return fail(KMERML_ERR_ARG, "row_stride_bytes must be a multiple of 16");
    return count_dense_host_impl(ctx, h_fasta, h_sizes, n_genomes, k_list, nk, min_record_len, flags, nullptr, 0, freq,
                                 freq_stride, h_totals, h_rows, row_stride_bytes);
}

static int compact_row_layout(const int* k_list, int nk, const uint8_t* h_row, RowSpec* row, WireLayout* lay) {
    if (!k_list || !h_row) return fail(KMERML_ERR_ARG, "null pointer argument");
    int kmax, kmin;
    int rc = build_row(k_list, nk, row, &kmax, &kmin);
    if (rc) return rc;
    uint32_t head[2];
    memcpy(head, h_row, 8);
    if (head[0] != WIRE_MAGIC) return fail(KMERML_ERR_ARG, "not a compact count row (bad header)");
    *lay = wire_layout(*row, true, head[1]);
    return KMERML_OK;
}

int kmerml_compact_row_overflowed(const int* k_list, int nk, const uint8_t* h_row) {
    RowSpec row;
    WireLayout lay;
    int rc = compact_row_layout(k_list, nk, h_row, &row, &lay);
    if (rc) return rc;
    uint32_t n_exc;
    memcpy(&n_exc, h_row + lay.exc_off, 4);
    return n_exc > NARROW_EXC_CAP ? 1 : 0;
}

uint64_t kmerml_compact_row_used_bytes(const int* k_list, int nk, const uint8_t* h_row) {
    RowSpec row;
    WireLayout lay;
    if (compact_row_layout(k_list, nk, h_row, &row, &lay)) return 0;
    return lay.bytes;
}

int kmerml_compact_expand(const int* k_list, int nk, const uint8_t* h_row, int ki, uint32_t* h_out) {
    if (!h_out || ki < 0 || ki >= nk) return fail(KMERML_ERR_ARG, "bad argument");
    RowSpec row;
    WireLayout lay;
    int rc = compact_row_layout(k_list, nk, h_row, &row, &lay);
    if (rc) return rc;
    const NarrowSpec& sp = lay.spec;
    const uint64_t n = 1ull << (2 * row.k[ki]);
    for (int i = 0; i < sp.n_small; i++)
        if (sp.small_src[i] == row.off[ki]) {
            memcpy(h_out, h_row + lay.small_off + sp.small_dst[i] * 4, (size_t)n * 4);
            return KMERML_OK;
        }
    for (int i = 0; i < sp.n; i++) {
        if (sp.src_off[i] != row.off[ki]) continue;
        uint32_t n_exc;
        memcpy(&n_exc, h_row + lay.exc_off, 4);
        if (n_exc > NARROW_EXC_CAP)
            return fail(KMERML_ERR_RANGE, "this genome's exception list overflowed: count it with kmerml_count_dense_host");
        if (sp.nibble[i]) widen_u4_to_u32(h_row + lay.narrow_off + sp.dst_off[i], h_out, (size_t)(n / 2));
        else widen_u8_to_u32(h_row + lay.narrow_off + sp.dst_off[i], h_out, (size_t)n);
        const uint32_t* e = reinterpret_cast<const uint32_t*>(h_row + lay.exc_off + 16);
        for (uint32_t j = 0; j < n_exc; j++)
            if (e[2 * j] >= row.off[ki] && e[2 * j] < row.off[ki] + n) h_out[e[2 * j] - row.off[ki]] = e[2 * j + 1];
        return KMERML_OK;
    }
    return fail(KMERML_ERR_ARG, "internal: level not found");
}

int kmerml_find_records(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint64_t* d_offsets, uint32_t cap,
                        uint32_t* h_count, void* stream) {
    if (!ctx || !h_count || (cap && !d_offsets)) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t s = (cudaStream_t)stream;
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.misc.ensure(256);
    if (rc) return rc;
    uint32_t* d_count = (uint32_t*)ws.misc.p;
    rc = launch_scan_records(d_fasta, nbytes, 0, (unsigned long long*)d_offsets, nullptr, cap, d_count, s);
    if (rc) return rc;
    KM_CUDA(cudaMemcpyAsync(h_count, d_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    return KMERML_OK;
}

int kmerml_records_short(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, const uint64_t* d_offsets,
                         uint32_t n, int min_record_len, uint8_t* d_is_short, void* stream) {
    if (!ctx || (n && (!d_offsets || !d_is_short))) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_record_short(d_fasta, nbytes, (const unsigned long long*)d_offsets, n, min_record_len, d_is_short,
                               (cudaStream_t)stream);
}

int kmerml_format_kmer_file(kmerml_ctx* ctx, int k, const uint32_t* d_counts, const uint32_t* d_first, unsigned flags,
                            uint64_t max_lines, uint8_t* d_text, uint64_t text_cap, uint64_t* h_text_len,
                            uint64_t* h_lines, void* stream) {
    if (!ctx || !d_counts || !d_first || !h_text_len || !h_lines) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (k < 1 || k > KMERML_MAX_DENSE_K) return fail(KMERML_ERR_ARG, "k out of range");
    if (text_cap && !d_text) return fail(KMERML_ERR_ARG, "d_text is null");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    max_lines = std::max<uint64_t>(max_lines, 1);
    int rc = ws.part.ensure(format_workspace_bytes(1ull << (2 * k), max_lines));
    if (rc) return rc;
    return run_format_dense(ws.part.p, k, d_counts, d_first, (flags & KMERML_FLAG_CANONICAL) != 0, max_lines, d_text,
                            text_cap, h_text_len, h_lines, (cudaStream_t)stream);
}

int kmerml_format_kmer_lines(kmerml_ctx* ctx, int k, const uint64_t* d_codes, const uint32_t* d_counts, uint64_t n,
                             uint8_t* d_text, uint64_t text_cap, uint64_t* h_text_len, void* stream) {
    if (!ctx || !h_text_len) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (n && (!d_codes || !d_counts)) return fail(KMERML_ERR_ARG, "null input pointer");
    if (text_cap && !d_text) return fail(KMERML_ERR_ARG, "d_text is null");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.part.ensure(format_workspace_bytes(1, std::max<uint64_t>(n, 1)));
    if (rc) return rc;
    return run_format_lines(ws.part.p, k, d_codes, d_counts, n, d_text, text_cap, h_text_len, (cudaStream_t)stream);
}

int kmerml_genome_stats(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint64_t* d_out, void* stream) {
    if (!ctx || !d_out || (nbytes && !d_fasta)) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_genome_stats(d_fasta, nbytes, (unsigned long long*)d_out, (cudaStream_t)stream);
}

int kmerml_parse_kmer_lines(kmerml_ctx* ctx, const uint8_t* d_text, const int64_t* d_line_end, uint64_t n_lines,
                            int64_t* d_value, int64_t* d_count, uint32_t* h_bad, void* stream) {
    if (!ctx || !h_bad || (n_lines && (!d_text || !d_line_end || !d_value || !d_count))) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.misc.ensure(256);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    rc = launch_parse_kmer_lines(d_text, (const long long*)d_line_end, n_lines, (long long*)d_value, (long long*)d_count,
                                 (unsigned int*)ws.misc.p, s);
    if (rc) return rc;
    KM_CUDA(cudaMemcpyAsync(h_bad, ws.misc.p, 4, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    return KMERML_OK;
}

int kmerml_feature_keys(kmerml_ctx* ctx, const int64_t* d_value, uint64_t n_rows, int64_t* d_keys, void* stream) {
    if (!ctx || (n_rows && (!d_value || !d_keys))) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_feature_keys((const long long*)d_value, n_rows, (long long*)d_keys, (cudaStream_t)stream);
}

int kmerml_feature_line_lengths(kmerml_ctx* ctx, const int64_t* d_value, const int64_t* d_count, const int64_t* d_class,
                                const int32_t* d_suffix_len, uint64_t n_rows, int64_t* d_len, void* stream) {
    if (!ctx || (n_rows && (!d_value || !d_count || !d_class || !d_suffix_len || !d_len))) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_feature_line_len((const long long*)d_value, (const long long*)d_count, (const long long*)d_class,
                                   (const int*)d_suffix_len, n_rows, (long long*)d_len, (cudaStream_t)stream);
}

int kmerml_feature_write_lines(kmerml_ctx* ctx, const int64_t* d_value, const int64_t* d_count, const int64_t* d_class,
                               const int64_t* d_suffix_off, const int32_t* d_suffix_len, const uint8_t* d_suffix_text,
                               const int64_t* d_line_off, uint64_t n_rows, uint8_t* d_out, void* stream) {
    if (!ctx || (n_rows && (!d_value || !d_count || !d_class || !d_suffix_off || !d_suffix_len || !d_line_off || !d_out)))
        return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_feature_write((const long long*)d_value, (const long long*)d_count, (const long long*)d_class,
                                (const long long*)d_suffix_off, (const int*)d_suffix_len, d_suffix_text,
                                (const long long*)d_line_off, n_rows, d_out, (cudaStream_t)stream);
}

int kmerml_count_stats(kmerml_ctx* ctx, const uint32_t* d_counts, uint64_t n_bins, uint64_t* d_out, void* stream) {
    if (!ctx || !d_out || (n_bins && !d_counts)) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.misc.ensure(count_stats_workspace());
    if (rc) return rc;
    return launch_count_stats(d_counts, n_bins, ws.misc.p, (unsigned long long*)d_out, (cudaStream_t)stream);
}

int kmerml_column_stats(kmerml_ctx* ctx, const void* d_x, int dtype, uint64_t stride, int n_rows, uint64_t m,
                        uint32_t* d_nnz, double* d_mean, double* d_var, void* stream) {
    if (!ctx || (m && (!d_x || !d_nnz || !d_mean || !d_var))) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (dtype < 0 || dtype > 2 || n_rows < 0 || stride < m) return fail(KMERML_ERR_ARG, "bad dtype / shape");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_column_stats(d_x, dtype, stride, n_rows, m, d_nnz, d_mean, d_var, (cudaStream_t)stream);
}

int kmerml_static_features(kmerml_ctx* ctx, int k, int compat, int32_t* d_out, void* stream) {
    if (!ctx || !d_out) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (k < 1 || k > KMERML_MAX_DENSE_K) return fail(KMERML_ERR_ARG, "k out of range");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_static_features(k, compat, d_out, (cudaStream_t)stream);
}

int kmerml_normalize_rows(kmerml_ctx* ctx, const uint32_t* d_counts, uint64_t counts_stride, const uint64_t* d_totals,
                          int n_rows, uint64_t m, float* d_out, uint64_t out_stride, void* stream) {
    if (!ctx || !d_counts || !d_totals || !d_out) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    return launch_normalize_rows(d_counts, counts_stride, d_totals, n_rows, m, d_out, out_stride, (cudaStream_t)stream);
}

int kmerml_pairwise_distance(kmerml_ctx* ctx, const void* d_x, int dtype, uint64_t stride, int n, uint64_t m,
                             int metric, float* d_out32, double* d_out64, void* stream) {
    if (!ctx || !d_x || (!d_out32 && !d_out64)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (dtype < 0 || dtype > 2 || metric < 0 || metric > 1 || n < 0) return fail(KMERML_ERR_ARG, "bad dtype / metric");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    // uint32 count rows: exact integer Gram matrix on the tensor cores (tcgen05 kind::i8)
    if (dtype == 1 && n > 0 && m >= 64 && m % 64 == 0) {
        int rc = ws.part.ensure(distance_rows_workspace(n, m));
        if (rc) return rc;
        return launch_distance_rows_tc((const uint32_t*)d_x, stride, n, m, 0, n, metric, ws.part.p, d_out32, d_out64,
                                       (cudaStream_t)stream);
    }
    int rc = ws.misc.ensure(256 + (size_t)n * n * sizeof(double));
    if (rc) return rc;
    double* d_gram = (double*)((uint8_t*)ws.misc.p + 256);
    return launch_pairwise(d_x, dtype, stride, n, m, metric, d_gram, d_out32, d_out64, (cudaStream_t)stream);
}

int kmerml_pairwise_distance_rows(kmerml_ctx* ctx, const uint32_t* d_counts, uint64_t stride, int n, uint64_t m,
                                  int row_begin, int row_end, int metric, float* d_out32, double* d_out64, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (metric < 0 || metric > 1 || n < 0 || row_begin < 0 || row_end > n || row_begin > row_end)
        return fail(KMERML_ERR_ARG, "bad metric / row range");
    if (row_begin == row_end) return KMERML_OK;
    if (!d_counts || (!d_out32 && !d_out64)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (m < 64 || m % 64) return fail(KMERML_ERR_ARG, "the row length must be a multiple of 64 (k >= 3)");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.part.ensure(distance_rows_workspace(n, m));
    if (rc) return rc;
    return launch_distance_rows_tc(d_counts, stride, n, m, row_begin, row_end, metric, ws.part.p, d_out32, d_out64,
                                   (cudaStream_t)stream);
}

int kmerml_count_planes(kmerml_ctx* ctx, const uint32_t* d_counts, uint64_t stride, int n, uint64_t m, uint8_t* d_planes,
                        uint64_t plane_stride, double* d_sumsq, uint32_t* d_max, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (n < 0 || stride < m || plane_stride < (uint64_t)n * m) return fail(KMERML_ERR_ARG, "bad shape / stride");
    if (n == 0) return KMERML_OK;
    if (!d_counts || !d_planes || !d_max) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    ctx->launches += 1;
    return launch_count_planes(d_counts, stride, n, m, d_planes, plane_stride, d_sumsq, d_max, (cudaStream_t)stream);
}

int kmerml_distance_rows_planes(kmerml_ctx* ctx, const uint8_t* d_planes, uint64_t plane_stride, int n_planes, int n,
                                uint64_t m, const double* d_sumsq, int row_begin, int row_end, int metric, float* d_out32,
                                double* d_out64, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (metric < 0 || metric > 1 || n < 0 || row_begin < 0 || row_end > n || row_begin > row_end)
        return fail(KMERML_ERR_ARG, "bad metric / row range");
    if (n_planes < 1 || n_planes > 4 || plane_stride < (uint64_t)n * m) return fail(KMERML_ERR_ARG, "bad planes");
    if (row_begin == row_end) return KMERML_OK;
    if (!d_planes || !d_sumsq || (!d_out32 && !d_out64)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (m < 64 || m % 64) return fail(KMERML_ERR_ARG, "the row length must be a multiple of 64 (k >= 3)");
    if (((uintptr_t)d_planes | plane_stride) & 15) return fail(KMERML_ERR_ARG, "planes must be 16-byte aligned");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.part.ensure(distance_rows_workspace(n, 0));
    if (rc) return rc;
    ctx->launches += 2;
    return launch_distance_rows_planes(d_planes, plane_stride, n_planes, n, m, d_sumsq, row_begin, row_end, metric, ws.part.p,
                                       d_out32, d_out64, (cudaStream_t)stream);
}

static int count_sparse_core(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin,
                             uint64_t range_end, int k, int min_record_len, unsigned flags, uint64_t* d_keys,
                             uint32_t* d_counts, uint32_t* d_first, uint64_t out_cap, uint64_t* h_unique,
                             uint64_t* h_windows, void* stream) {
    if (!ctx || !h_unique || !h_windows) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (nbytes && !d_fasta) return fail(KMERML_ERR_ARG, "d_fasta is null");
    if (out_cap && (!d_keys || !d_counts)) return fail(KMERML_ERR_ARG, "null output pointer");
    if (nbytes >= 0xFFFFFFFFull) return fail(KMERML_ERR_RANGE, "genome too large for 32-bit offsets");
    if ((uintptr_t)d_fasta & 15) return fail(KMERML_ERR_ARG, "device pointers must be 16-byte aligned");
    if (range_begin > range_end || range_end > nbytes) return fail(KMERML_ERR_ARG, "byte range outside the file");
    if (range_begin % KMERML_SPARSE_RANGE_ALIGN || (range_end % KMERML_SPARSE_RANGE_ALIGN && range_end != nbytes))
        return fail(KMERML_ERR_ARG, "byte range must be aligned to KMERML_SPARSE_RANGE_ALIGN");
    int min_rec = min_record_len > 0 ? min_record_len : k;
    if (min_rec < k) return fail(KMERML_ERR_ARG, "min_record_len must be >= k");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    // at most one window ends at every byte of the range; the slice table covers the whole file
    const uint64_t cap = std::max<uint64_t>(range_end - range_begin, 1);
    int rc = ws.part.ensure(sparse_workspace_bytes(cap));
    if (rc) return rc;
    DevWalk w;
    if ((rc = put_single_walk(ws, d_fasta, nbytes, SPARSE_SLICE_BYTES, SPARSE_TILE_BYTES, (cudaStream_t)stream, &w))) return rc;
    rc = run_sparse_in(ws.part.p, d_fasta, w.genomes, w.slices, w.n_slices, range_begin, range_end, k, min_rec,
                       (flags & KMERML_FLAG_CANONICAL) != 0, cap, d_keys, d_counts, d_first, out_cap, h_unique,
                       h_windows, &ctx->sparse_pending, (cudaStream_t)stream);
    ctx->sparse_pending.cap = cap;
    ctx->sparse_pending.workspace = ws.part.p;
    return rc;
}

int kmerml_emit_sparse_range(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin,
                             uint64_t range_end, int k, int min_record_len, unsigned flags, int owner_bits, uint64_t* d_keys,
                             uint32_t* d_ends, uint64_t out_cap, uint64_t* h_windows, uint64_t* h_owner_counts, void* stream) {
    if (!ctx || !h_windows || !h_owner_counts) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (owner_bits < 0 || owner_bits > 5 || owner_bits > 2 * k) return fail(KMERML_ERR_ARG, "owner_bits must be in 0..5");
    if (nbytes && !d_fasta) return fail(KMERML_ERR_ARG, "d_fasta is null");
    if (out_cap && (!d_keys || !d_ends)) return fail(KMERML_ERR_ARG, "null output pointer");
    if (nbytes >= 0xFFFFFFFFull) return fail(KMERML_ERR_RANGE, "genome too large for 32-bit offsets");
    if ((uintptr_t)d_fasta & 15) return fail(KMERML_ERR_ARG, "device pointers must be 16-byte aligned");
    if (range_begin > range_end || range_end > nbytes) return fail(KMERML_ERR_ARG, "byte range outside the file");
    if (range_begin % KMERML_SPARSE_RANGE_ALIGN || (range_end % KMERML_SPARSE_RANGE_ALIGN && range_end != nbytes))
        return fail(KMERML_ERR_ARG, "byte range must be aligned to KMERML_SPARSE_RANGE_ALIGN");
    int min_rec = min_record_len > 0 ? min_record_len : k;
    if (min_rec < k) return fail(KMERML_ERR_ARG, "min_record_len must be >= k");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    const uint64_t cap = std::max<uint64_t>(range_end - range_begin, 1);
    int rc = ws.part.ensure(sparse_workspace_bytes(cap));
    if (rc) return rc;
    ctx->sparse_pending.valid = false;
    DevWalk w;
    if ((rc = put_single_walk(ws, d_fasta, nbytes, SPARSE_SLICE_BYTES, SPARSE_TILE_BYTES, (cudaStream_t)stream, &w))) return rc;
    return run_sparse_emit_by_owner(ws.part.p, d_fasta, w.genomes, w.slices, w.n_slices, range_begin, range_end, k, min_rec,
                                    (flags & KMERML_FLAG_CANONICAL) != 0, owner_bits, cap, d_keys, d_ends, out_cap, h_windows,
                                    h_owner_counts, (cudaStream_t)stream);
}

int kmerml_reduce_sparse_windows(kmerml_ctx* ctx, int sort_bits, const uint64_t* d_keys, const uint32_t* d_ends, uint64_t n,
                                 uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                                 uint64_t* h_unique, void* stream) {
    if (!ctx || !h_unique) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (sort_bits < 1 || sort_bits > 64) return fail(KMERML_ERR_ARG, "sort_bits must be in 1..64");
    if (n && (!d_keys || !d_ends)) return fail(KMERML_ERR_ARG, "null input pointer");
    if (out_cap && (!d_keys_out || !d_counts_out)) return fail(KMERML_ERR_ARG, "null output pointer");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    const uint64_t cap = std::max<uint64_t>(n, 1);
    int rc = ws.part.ensure(sparse_workspace_bytes(cap));
    if (rc) return rc;
    rc = run_sparse_reduce_windows(ws.part.p, sort_bits, d_keys, d_ends, n, d_keys_out, d_counts_out, d_first_out, out_cap,
                                   h_unique, &ctx->sparse_pending, (cudaStream_t)stream);
    ctx->sparse_pending.cap = cap;
    ctx->sparse_pending.workspace = ws.part.p;
    return rc;
}

int kmerml_sparse_fetch(kmerml_ctx* ctx, uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first, uint64_t out_cap,
                        void* stream) {
    if (!ctx || !d_keys || !d_counts) return fail(KMERML_ERR_ARG, "null pointer argument");
    const SparsePending& p = ctx->sparse_pending;
    if (!p.valid || p.workspace != ctx->ws[0].part.p)
        return fail(KMERML_ERR_ARG, "no sparse result to fetch (another call has used the workspace since)");
    if (out_cap < p.nu) return fail(KMERML_ERR_ARG, "outputs smaller than the number of distinct k-mers");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return sparse_fetch(ctx->ws[0].part.p, p, d_keys, d_counts, d_first, (cudaStream_t)stream);
}

int kmerml_count_sparse(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, int k, int min_record_len,
                        unsigned flags, uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first, uint64_t out_cap,
                        uint64_t* h_unique, uint64_t* h_windows, void* stream) {
    return count_sparse_core(ctx, d_fasta, nbytes, 0, nbytes, k, min_record_len, flags, d_keys, d_counts, d_first, out_cap,
                             h_unique, h_windows, stream);
}

int kmerml_count_sparse_range(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint64_t range_begin,
                              uint64_t range_end, int k, int min_record_len, unsigned flags, uint64_t* d_keys,
                              uint32_t* d_counts, uint32_t* d_first, uint64_t out_cap, uint64_t* h_unique,
                              uint64_t* h_windows, void* stream) {
    return count_sparse_core(ctx, d_fasta, nbytes, range_begin, range_end, k, min_record_len, flags, d_keys, d_counts,
                             d_first, out_cap, h_unique, h_windows, stream);
}

int kmerml_merge_sparse(kmerml_ctx* ctx, int k, const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first,
                        uint64_t n, uint64_t* d_keys_out, uint32_t* d_counts_out, uint32_t* d_first_out, uint64_t out_cap,
                        uint64_t* h_unique, void* stream) {
    if (!ctx || !h_unique) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (n && (!d_keys || !d_counts)) return fail(KMERML_ERR_ARG, "null input pointer");
    if (out_cap && (!d_keys_out || !d_counts_out)) return fail(KMERML_ERR_ARG, "null output pointer");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    int rc = ws.part.ensure(merge_workspace_bytes(std::max<uint64_t>(n, 1)));
    if (rc) return rc;
    return run_merge_sparse(ws.part.p, k, d_keys, d_counts, d_first, n, d_keys_out, d_counts_out, d_first_out, out_cap,
                            h_unique, (cudaStream_t)stream);
}

int kmerml_first_occurrence(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, int k, int min_record_len,
                            uint32_t* d_first, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (k < 1 || k > KMERML_MAX_DENSE_K) return fail(KMERML_ERR_ARG, "k out of range");
    if (!d_first || (nbytes && !d_fasta)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (((uintptr_t)d_fasta & 15)) return fail(KMERML_ERR_ARG, "device pointers must be 16-byte aligned");
    if (nbytes >= 0xFFFFFFFFull) return fail(KMERML_ERR_RANGE, "genome too large for 32-bit offsets");
    int min_rec = min_record_len > 0 ? min_record_len : k;
    if (min_rec < k) return fail(KMERML_ERR_ARG, "min_record_len must be >= k");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t s = (cudaStream_t)stream;
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    KM_CUDA(cudaMemsetAsync(d_first, 0xFF, (size_t)(1ull << (2 * k)) * 4, s));
    if (!nbytes) return KMERML_OK;
    DevWalk w;
    int rc = put_single_walk(ws, d_fasta, nbytes, atomic_slice_bytes(ctx->sm_count, nbytes), TILE_BYTES, s, &w);
    if (rc) return rc;
    return launch_first_occurrence(d_fasta, w.genomes, w.slices, w.n_slices, k, min_rec, d_first, s);
}

// ---- MinHash sketches (sketch.cu) ----
// First threshold of a genome: ~3 s windows hash below it (windows <= bytes); every window when that is all of them.
static uint64_t sketch_first_tau(uint64_t bytes, int s) {
    const unsigned __int128 want = (unsigned __int128)3 * (unsigned)s;
    if (want >= bytes) return ~0ull;
    return (uint64_t)((want << 64) / bytes);
}

// Region of a genome at threshold tau: twice the survivors expected, one slot per byte at most (>= its windows).
static uint64_t sketch_region(uint64_t bytes, uint64_t tau) {
    if (tau == ~0ull) return bytes;
    const uint64_t expect = (uint64_t)(((unsigned __int128)bytes * tau) >> 64);
    return std::min<uint64_t>(bytes, 2 * expect + 1024);
}

constexpr uint64_t SKETCH_ROUND_SLOTS = 1ull << 28;     // survivor slots of one round (2 GiB, twice: sort in / out)

// One emit round of sketch_rounds, as the caller's stage sees it: the genomes h_active[0 .. n_active) (buffer order;
// the same on the device at d_active) with their thresholds, regions and survivor counts at d_sg[genome], the
// survivors of each region sorted into d_sorted, d_seg the sort's 2 n_active int segment bounds (begins | ends),
// n_active status words (device d_status, pinned host h_status) and the stage's own scratch.
struct SketchRound {
    int n_active;
    const int* h_active;
    const int* d_active;
    const SketchGenome* d_sg;
    const int* d_seg;
    uint64_t slots;
    const uint64_t* d_sorted;
    void* scratch;
    uint32_t* d_status;
    uint32_t* h_status;
};

// The round loop of the sketch calls.  Genomes still pending, in buffer order, are packed into rounds of at most
// SKETCH_ROUND_SLOTS survivor slots (at least one genome); a round walks their slices with sketch_emit_kernel (genome
// g: threshold tau[g], region of cap[g] slots) and sorts every region.  `stage_bytes(slots, n_active)` is the scratch
// the caller's stage needs; `stage` launches its selection, waits for it and lists the genomes to run again, for
// which it has set tau and cap anew.
static int sketch_rounds(kmerml_ctx* ctx, const uint8_t* d_fasta, const uint64_t* h_offsets, int n, int k, int min_rec,
                         bool canonical, uint64_t seed, std::vector<uint64_t>& tau, std::vector<uint64_t>& cap,
                         const std::function<size_t(uint64_t, int)>& stage_bytes,
                         const std::function<int(const SketchRound&, std::vector<int>&)>& stage, cudaStream_t s) {
    // the slice table of a round holds at most the slices of every genome
    std::vector<uint64_t> slice_bytes(n, SPARSE_SLICE_BYTES);
    std::vector<Slice> plan;
    std::vector<uint32_t> first;
    int rc = plan_slices(h_offsets, n, slice_bytes.data(), SPARSE_TILE_BYTES, 0, 0, plan, first);
    if (rc) return rc;
    // tables: offsets | genomes | stats | sketch genomes | active | segments | status | slices
    Tables t{ctx->ws[0]};
    Walk walk(t, n);
    const size_t at_sg = t.take((size_t)n * sizeof(SketchGenome)), at_active = t.take((size_t)n * 4);
    const size_t at_seg = t.take((size_t)n * 8), at_status = t.take((size_t)n * 4);
    walk.take_slices(t, plan.size() - 1);
    if ((rc = t.open()) || (rc = put_walk(t, walk, d_fasta, h_offsets, nullptr, s))) return rc;
    const GenomeDev* d_genomes = t.dev<GenomeDev>(walk.genomes);
    const Slice* d_slices = t.dev<Slice>(walk.slices);
    Workspace& ws = ctx->ws[0];

    std::vector<int> pending(n);
    for (int g = 0; g < n; g++) pending[g] = g;
    while (!pending.empty()) {
        // one round: the pending genomes (in buffer order) whose regions fit SKETCH_ROUND_SLOTS, at least one
        SketchGenome* h_sg = t.fill<SketchGenome>(at_sg, (size_t)n * sizeof(SketchGenome));
        int* h_active = t.host<int>(at_active);
        memset(h_sg, 0, (size_t)n * sizeof(SketchGenome));
        std::fill(slice_bytes.begin(), slice_bytes.end(), 0);
        int n_round = 0;
        uint64_t slots = 0;
        for (int g : pending) {
            if (n_round && slots + cap[g] > SKETCH_ROUND_SLOTS) break;
            if (slots + cap[g] > 0x7fffffffull)
                return fail(KMERML_ERR_RANGE, "a genome's sketch region exceeds 2^31 slots");
            h_sg[g].tau = tau[g];
            h_sg[g].region = slots;
            h_sg[g].cap = cap[g];
            h_active[n_round++] = g;
            slots += cap[g];
            slice_bytes[g] = SPARSE_SLICE_BYTES;
        }
        t.fill<int>(at_active, (size_t)n_round * 4);
        if ((rc = plan_slices(h_offsets, n, slice_bytes.data(), SPARSE_TILE_BYTES, 0, 0, plan, first))) return rc;
        const size_t region_bytes = align_up(std::max<uint64_t>(slots, 1) * 8, 256);
        const size_t temp_bytes = align_up(sketch_sort_temp_bytes((int)slots, n_round), 256);
        if ((rc = ws.part.ensure(2 * region_bytes + temp_bytes + stage_bytes(slots, n_round)))) return rc;
        uint64_t* d_regions = (uint64_t*)ws.part.p;
        uint64_t* d_sorted = (uint64_t*)((uint8_t*)ws.part.p + region_bytes);
        void* d_temp = (uint8_t*)ws.part.p + 2 * region_bytes;
        {
            Prof pr(ctx, s, 3, 6);      // the three slice-table kernels, emit, segments, sort
            rc = put_walk(t, walk, d_fasta, nullptr, &plan, s);
            if (!rc) rc = launch_sketch_emit(d_fasta, d_genomes, d_slices, walk.n_slices, k, min_rec, canonical, seed, t.dev<SketchGenome>(at_sg),
                                             d_regions, s);
            if (!rc) rc = launch_sketch_sort(t.dev<SketchGenome>(at_sg), t.dev<int>(at_active), n_round, t.dev<int>(at_seg), (int)slots,
                                             d_regions, d_sorted, d_temp, temp_bytes, s);
        }
        if (rc) return rc;
        const SketchRound round{n_round, h_active, t.dev<int>(at_active), t.dev<SketchGenome>(at_sg), t.dev<int>(at_seg), slots,
                                d_sorted, (uint8_t*)d_temp + temp_bytes, t.dev<uint32_t>(at_status), t.host<uint32_t>(at_status)};
        std::vector<int> next;
        if ((rc = stage(round, next))) return rc;
        next.insert(next.end(), pending.begin() + n_round, pending.end());
        std::sort(next.begin(), next.end());            // the slice table stays in buffer order
        pending.swap(next);
    }
    return KMERML_OK;
}

static int sketch_batch_core(kmerml_ctx* ctx, const uint8_t* d_fasta, const uint64_t* h_offsets, int n, int k, int min_rec,
                             bool canonical, int sketch_size, uint64_t seed, uint64_t* d_sketches, uint64_t stride,
                             uint32_t* d_filled, cudaStream_t s) {
    std::vector<uint64_t> tau(n), cap(n);
    for (int g = 0; g < n; g++) {
        const uint64_t bytes = h_offsets[g + 1] - h_offsets[g];
        tau[g] = sketch_first_tau(bytes, sketch_size);
        cap[g] = sketch_region(bytes, tau[g]);
    }
    auto select = [&](const SketchRound& r, std::vector<int>& again) {
        {
            Prof pr(ctx, s, 3, 1);
            int rc = launch_sketch_select(r.d_sg, r.d_active, r.n_active, r.d_sorted, sketch_size, d_sketches, stride,
                                          d_filled, r.d_status, s);
            if (rc) return rc;
        }
        KM_CUDA(cudaMemcpyAsync(r.h_status, r.d_status, (size_t)r.n_active * 4, cudaMemcpyDeviceToHost, s));
        KM_CUDA(cudaStreamSynchronize(s));
        // run again: too few distinct hashes below tau -> 16 tau (saturating at every window); overflow -> one slot
        // per byte.  Every window with one slot per byte cannot fail, so the loop ends.
        for (int i = 0; i < r.n_active; i++) {
            const int g = r.h_active[i];
            const uint64_t bytes = h_offsets[g + 1] - h_offsets[g];
            if (r.h_status[i] == SKETCH_MORE) {
                tau[g] = tau[g] > ~0ull / 16 ? ~0ull : tau[g] * 16;
                cap[g] = sketch_region(bytes, tau[g]);
            } else if (r.h_status[i] == SKETCH_OVERFLOW) {
                cap[g] = bytes;
            } else {
                continue;
            }
            again.push_back(g);
        }
        return KMERML_OK;
    };
    return sketch_rounds(ctx, d_fasta, h_offsets, n, k, min_rec, canonical, seed, tau, cap,
                         [](uint64_t, int) { return (size_t)0; }, select, s);
}

// Grows `b` to `bytes`, keeping its first `used` bytes (`s` is idle when this is called).
static int grow_keeping(DevBuf& b, size_t used, size_t bytes, cudaStream_t s) {
    if (bytes <= b.cap) return KMERML_OK;
    DevBuf nb;
    int rc = nb.ensure(std::max(bytes, b.cap * 2));
    if (rc) return rc;
    if (used) KM_CUDA(cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, s));
    KM_CUDA(cudaStreamSynchronize(s));
    b.release();
    b = nb;
    return KMERML_OK;
}

// Scaled sketches: the rounds of sketch_rounds with tau = T for every genome.  After each round the distinct values of
// the genomes that did not overflow are appended to ctx->fmh_kept; at the end the CSR offsets and the gather into the
// caller's buffer put them in genome order.  With `abundance` each kept value's run length in the sorted round is
// appended to ctx->fmh_abund in the same places.
static int fmh_batch_core(kmerml_ctx* ctx, const uint8_t* d_fasta, const uint64_t* h_offsets, int n, int k, int min_rec,
                          bool canonical, bool abundance, uint64_t scale, uint64_t seed, uint64_t* d_hashes,
                          uint64_t out_cap, uint64_t* d_offsets, uint64_t* h_total, cudaStream_t s) {
    const uint64_t T = ~0ull / scale;
    const auto too_large = [&](int g) {
        return fail(KMERML_ERR_RANGE, "genome " + std::to_string(g) + ": its k-mers at or below the threshold of scale " +
                                          std::to_string(scale) + " may exceed 2^31 - 1; use a larger scale");
    };
    std::vector<uint64_t> tau(n, T), cap(n), begin(n, 0), size(n, 0);
    for (int g = 0; g < n; g++) {
        cap[g] = sketch_region(h_offsets[g + 1] - h_offsets[g], T);
        if (cap[g] > 0x7fffffffull) return too_large(g);
    }
    ctx->fmh_n = -1;
    ctx->fmh_has_abund = false;
    uint64_t kept = 0;                                 // values in ctx->fmh_kept
    auto scratch = [](uint64_t slots, int n_active) {
        return 2 * align_up(std::max<uint64_t>(slots, 1) * 4, 256) + align_up(fmh_scan_temp_bytes((int)slots), 256) +
               (size_t)n_active * sizeof(FmhRoundGenome);
    };
    auto distinct = [&](const SketchRound& r, std::vector<int>& again) {
        const size_t flag_bytes = align_up(std::max<uint64_t>(r.slots, 1) * 4, 256);
        const size_t temp_bytes = align_up(fmh_scan_temp_bytes((int)r.slots), 256);
        uint32_t* d_flags = (uint32_t*)r.scratch;
        uint32_t* d_pos = (uint32_t*)((uint8_t*)r.scratch + flag_bytes);
        void* d_temp = (uint8_t*)r.scratch + 2 * flag_bytes;
        FmhRoundGenome* d_out = (FmhRoundGenome*)((uint8_t*)d_temp + temp_bytes);
        {
            Prof pr(ctx, s, 3, 3);
            int rc = launch_fmh_distinct(r.d_sg, r.d_active, r.n_active, r.d_seg, (int)r.slots, r.d_sorted, d_flags, d_pos,
                                         d_temp, temp_bytes, d_out, s);
            if (rc) return rc;
        }
        std::vector<FmhRoundGenome> out(r.n_active);
        KM_CUDA(cudaMemcpyAsync(out.data(), d_out, out.size() * sizeof(FmhRoundGenome), cudaMemcpyDeviceToHost, s));
        KM_CUDA(cudaStreamSynchronize(s));
        uint64_t round_kept = 0;
        for (int i = 0; i < r.n_active; i++) {
            const int g = r.h_active[i];
            if (out[i].count > cap[g]) {               // overflow: the cursor counted every survivor
                if (out[i].count > 0x7fffffffull) return too_large(g);
                cap[g] = out[i].count;
                again.push_back(g);
                continue;
            }
            begin[g] = kept + out[i].first;
            size[g] = out[i].distinct;
            round_kept += out[i].distinct;
        }
        if (!round_kept) return KMERML_OK;
        int rc = grow_keeping(ctx->fmh_kept, kept * 8, (kept + round_kept) * 8, s);
        if (!rc && abundance) rc = grow_keeping(ctx->fmh_abund, kept * 4, (kept + round_kept) * 4, s);
        if (!rc) {
            Prof pr(ctx, s, 3, abundance ? 2 : 1);
            rc = launch_fmh_scatter(r.d_sorted, d_flags, d_pos, (int)r.slots, (uint64_t*)ctx->fmh_kept.p + kept, s);
            if (!rc && abundance)
                rc = launch_fmh_abundance(d_flags, d_pos, r.d_seg, r.n_active, (int)r.slots,
                                          (uint32_t*)ctx->fmh_abund.p + kept, s);
        }
        kept += round_kept;
        return rc;
    };
    int rc = sketch_rounds(ctx, d_fasta, h_offsets, n, k, min_rec, canonical, seed, tau, cap, scratch, distinct, s);
    if (rc) return rc;
    // the index: begin | CSR offsets, uploaded from pageable memory (the call is synchronous)
    std::vector<uint64_t> index(2 * (size_t)n + 1);
    for (int g = 0; g < n; g++) {
        index[g] = begin[g];
        index[n + g + 1] = index[n + g] + size[g];
    }
    if ((rc = ctx->fmh_index.ensure(index.size() * 8))) return rc;
    KM_CUDA(cudaMemcpyAsync(ctx->fmh_index.p, index.data(), index.size() * 8, cudaMemcpyHostToDevice, s));
    KM_CUDA(cudaStreamSynchronize(s));
    ctx->fmh_n = n;
    ctx->fmh_has_abund = abundance;
    ctx->fmh_total = index[2 * (size_t)n];
    *h_total = ctx->fmh_total;
    KM_CUDA(cudaMemcpyAsync(d_offsets, (uint64_t*)ctx->fmh_index.p + n, (size_t)(n + 1) * 8, cudaMemcpyDeviceToDevice, s));
    if (ctx->fmh_total <= out_cap) {
        ctx->launches += 1;
        rc = launch_fmh_gather((const uint64_t*)ctx->fmh_kept.p, (const uint64_t*)ctx->fmh_index.p,
                               (const uint64_t*)ctx->fmh_index.p + n, n, ctx->fmh_total, d_hashes, s);
    }
    if (!rc) KM_CUDA(cudaStreamSynchronize(s));
    return rc;
}

int kmerml_sketch_batch(kmerml_ctx* ctx, const uint8_t* d_fasta, const uint64_t* h_offsets, int n_genomes, int k,
                        int min_record_len, unsigned flags, int sketch_size, uint64_t seed, uint64_t* d_sketches,
                        uint64_t sketch_stride, uint32_t* d_filled, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (sketch_size < 1 || sketch_size > KMERML_SKETCH_MAX)
        return fail(KMERML_ERR_ARG, "sketch_size must be in 1.." + std::to_string(KMERML_SKETCH_MAX));
    if (sketch_stride < (uint64_t)sketch_size) return fail(KMERML_ERR_ARG, "sketch_stride must be >= sketch_size");
    if (n_genomes < 0) return fail(KMERML_ERR_ARG, "n_genomes < 0");
    const int min_rec = min_record_len > 0 ? min_record_len : k;
    if (min_rec < k) return fail(KMERML_ERR_ARG, "min_record_len must be >= k");
    if (n_genomes == 0) return KMERML_OK;
    if (!h_offsets || !d_sketches || !d_filled) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (int rc = check_batch(d_fasta, h_offsets, n_genomes, false)) return rc;
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return sketch_batch_core(ctx, d_fasta, h_offsets, n_genomes, k, min_rec, (flags & KMERML_FLAG_CANONICAL) != 0,
                             sketch_size, seed, d_sketches, sketch_stride, d_filled, (cudaStream_t)stream);
}

int kmerml_sketch_distance_rows(kmerml_ctx* ctx, const uint64_t* d_sketches, uint64_t sketch_stride, const uint32_t* d_filled,
                                int n, int sketch_size, int k, int row_begin, int row_end, int metric, float* d_out32,
                                double* d_out64, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (sketch_size < 1 || sketch_size > KMERML_SKETCH_MAX)
        return fail(KMERML_ERR_ARG, "sketch_size must be in 1.." + std::to_string(KMERML_SKETCH_MAX));
    if (sketch_stride < (uint64_t)sketch_size) return fail(KMERML_ERR_ARG, "sketch_stride must be >= sketch_size");
    if (metric != KMERML_SKETCH_METRIC_MASH && metric != KMERML_SKETCH_METRIC_JACCARD)
        return fail(KMERML_ERR_ARG, "unknown sketch metric");
    if (n < 0 || row_begin < 0 || row_end > n || row_begin > row_end) return fail(KMERML_ERR_ARG, "bad row range");
    if (row_begin == row_end) return KMERML_OK;
    if (!d_sketches || !d_filled || (!d_out32 && !d_out64)) return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    ctx->launches += 1;
    return launch_sketch_distance(d_sketches, sketch_stride, d_filled, n, sketch_size, k, row_begin, row_end, metric,
                                  d_out32, d_out64, (cudaStream_t)stream);
}

int kmerml_fmh_batch(kmerml_ctx* ctx, const uint8_t* d_fasta, const uint64_t* h_offsets, int n_genomes, int k,
                     int min_record_len, unsigned flags, uint64_t scale, uint64_t seed, uint64_t* d_hashes, uint64_t out_cap,
                     uint64_t* d_sketch_offsets, uint64_t* h_total, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (scale < 1) return fail(KMERML_ERR_ARG, "scale must be >= 1");
    if (n_genomes < 0) return fail(KMERML_ERR_ARG, "n_genomes < 0");
    const int min_rec = min_record_len > 0 ? min_record_len : k;
    if (min_rec < k) return fail(KMERML_ERR_ARG, "min_record_len must be >= k");
    if (!h_offsets || !d_sketch_offsets || !h_total || (out_cap && !d_hashes)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (int rc = check_batch(d_fasta, h_offsets, n_genomes, false)) return rc;
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return fmh_batch_core(ctx, d_fasta, h_offsets, n_genomes, k, min_rec, (flags & KMERML_FLAG_CANONICAL) != 0,
                          (flags & KMERML_FLAG_FMH_ABUNDANCE) != 0, scale, seed, d_hashes, out_cap, d_sketch_offsets,
                          h_total, (cudaStream_t)stream);
}

int kmerml_fmh_fetch(kmerml_ctx* ctx, uint64_t* d_hashes, uint64_t out_cap, uint64_t* d_sketch_offsets, void* stream) {
    if (!ctx || !d_sketch_offsets || (out_cap && !d_hashes)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (ctx->fmh_n < 0) return fail(KMERML_ERR_ARG, "no scaled-sketch result to fetch");
    if (out_cap < ctx->fmh_total) return fail(KMERML_ERR_ARG, "out_cap is smaller than the total of the sketches");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    cudaStream_t s = (cudaStream_t)stream;
    const int n = ctx->fmh_n;
    const uint64_t* index = (const uint64_t*)ctx->fmh_index.p;
    KM_CUDA(cudaMemcpyAsync(d_sketch_offsets, index + n, (size_t)(n + 1) * 8, cudaMemcpyDeviceToDevice, s));
    ctx->launches += 1;
    int rc = launch_fmh_gather((const uint64_t*)ctx->fmh_kept.p, index, index + n, n, ctx->fmh_total, d_hashes, s);
    if (!rc) KM_CUDA(cudaStreamSynchronize(s));
    return rc;
}

int kmerml_fmh_compare(kmerml_ctx* ctx, const uint64_t* d_q_hashes, const uint64_t* d_q_offsets, int n_q,
                       const uint64_t* d_r_hashes, const uint64_t* d_r_offsets, int n_r, int k, int metric,
                       uint32_t* d_intersections, float* d_out32, double* d_out64, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (k < 1 || k > KMERML_MAX_K) return fail(KMERML_ERR_ARG, "k must be in 1..32");
    if (metric < KMERML_FMH_CONTAINMENT || metric > KMERML_FMH_MAX_CONTAINMENT_ANI)
        return fail(KMERML_ERR_ARG, "unknown scaled-sketch metric");
    if (n_q < 0 || n_r < 0) return fail(KMERML_ERR_ARG, "n_q and n_r must be >= 0");
    if (!n_q || !n_r) return KMERML_OK;
    if (!d_q_hashes || !d_q_offsets || !d_r_hashes || !d_r_offsets || (!d_intersections && !d_out32 && !d_out64))
        return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    // workspace: the reference chunk table | the intersections when the caller does not want them
    const size_t table = align_up(fmh_compare_workspace(n_r), 256);
    int rc = ws.misc.ensure(table + (d_intersections ? 0 : (size_t)n_q * n_r * 4));
    if (rc) return rc;
    uint32_t* inter = d_intersections ? d_intersections : (uint32_t*)((uint8_t*)ws.misc.p + table);
    ctx->launches += 3;
    return launch_fmh_compare(d_q_hashes, d_q_offsets, n_q, d_r_hashes, d_r_offsets, n_r, k, metric, ctx->sm_count, ws.misc.p,
                              inter, d_out32, d_out64, (cudaStream_t)stream);
}

int kmerml_fmh_fetch_abundances(kmerml_ctx* ctx, uint32_t* d_abundances, uint64_t out_cap, void* stream) {
    if (!ctx || (out_cap && !d_abundances)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (ctx->fmh_n < 0 || !ctx->fmh_has_abund)
        return fail(KMERML_ERR_ARG, "no scaled-sketch result made with KMERML_FLAG_FMH_ABUNDANCE to fetch");
    if (out_cap < ctx->fmh_total) return fail(KMERML_ERR_ARG, "out_cap is smaller than the total of the sketches");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    cudaStream_t s = (cudaStream_t)stream;
    const int n = ctx->fmh_n;
    const uint64_t* index = (const uint64_t*)ctx->fmh_index.p;
    ctx->launches += 1;
    int rc = launch_fmh_gather((const uint32_t*)ctx->fmh_abund.p, index, index + n, n, ctx->fmh_total, d_abundances, s);
    if (!rc) KM_CUDA(cudaStreamSynchronize(s));
    return rc;
}

int kmerml_fmh_compare_weighted(kmerml_ctx* ctx, const uint64_t* d_q_hashes, const uint64_t* d_q_offsets,
                                const uint32_t* d_q_abundances, int n_q, const uint64_t* d_r_hashes,
                                const uint64_t* d_r_offsets, const uint32_t* d_r_abundances, int n_r, int metric,
                                uint64_t* d_numerators, float* d_out32, double* d_out64, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (metric != KMERML_FMH_WEIGHTED_CONTAINMENT && metric != KMERML_FMH_ANGULAR_SIMILARITY)
        return fail(KMERML_ERR_ARG, "unknown weighted scaled-sketch metric");
    if (n_q < 0 || n_r < 0) return fail(KMERML_ERR_ARG, "n_q and n_r must be >= 0");
    if (!n_q || !n_r) return KMERML_OK;
    if (!d_q_hashes || !d_q_offsets || !d_q_abundances || !d_r_hashes || !d_r_offsets ||
        (metric == KMERML_FMH_ANGULAR_SIMILARITY && !d_r_abundances) || (!d_numerators && !d_out32 && !d_out64))
        return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    // workspace: the reference chunk table and the per-sketch sums | the numerators when the caller does not want them
    const size_t table = align_up(fmh_compare_weighted_workspace(n_q, n_r), 256);
    int rc = ws.misc.ensure(table + (d_numerators ? 0 : (size_t)n_q * n_r * 8));
    if (rc) return rc;
    unsigned long long* num = d_numerators ? (unsigned long long*)d_numerators
                                           : (unsigned long long*)((uint8_t*)ws.misc.p + table);
    ctx->launches += 2 + ((d_out32 || d_out64) ? (metric == KMERML_FMH_ANGULAR_SIMILARITY ? 3 : 2) : 0);
    return launch_fmh_compare_weighted(d_q_hashes, d_q_offsets, d_q_abundances, n_q, d_r_hashes, d_r_offsets,
                                       d_r_abundances, n_r, metric, ctx->sm_count, ws.misc.p, num, d_out32, d_out64,
                                       (cudaStream_t)stream);
}

// Gather: x = |Q n R| for every pair (launch_fmh_compare), the candidate references (x >= threshold for some query)
// copied into a compact CSR in reference order, then rounds in lockstep over every running query: select (with the
// last round's subtraction fused), remove (the hashes the pick takes, as a sorted CSR S_t) and subtract
// (launch_fmh_compare of S_t against the candidates).  The host reads the number of picks after each select and
// stops when there were none or max_matches rounds have run.  With query abundances (d_qa; NULL for
// kmerml_fmh_gather) the remove step also sums S_t's abundances and a segmented sort gives their median; it then runs
// in the last round too, so the last recorded match gets its statistics.
static int fmh_gather_core(kmerml_ctx* ctx, const uint64_t* d_qh, const uint64_t* d_q_off, int n_q, const uint64_t* d_rh,
                           const uint64_t* d_r_off, int n_r, uint32_t threshold, int max_matches, int32_t* d_n_matches,
                           int32_t* d_ref, uint32_t* d_unique, uint32_t* d_inter, uint32_t* d_rem, const uint32_t* d_qa,
                           uint64_t* d_uw, uint64_t* d_usq, double* d_med, cudaStream_t s) {
    Workspace& ws = ctx->ws[0];
    KM_CUDA(cudaMemsetAsync(d_n_matches, 0, (size_t)n_q * 4, s));
    if (!n_r) {
        KM_CUDA(cudaStreamSynchronize(s));
        return KMERML_OK;
    }
    // ws.part: x (n_q x n_r) | the chunk table of launch_fmh_compare (n_r >= the candidates) | candidate flags
    const size_t x_bytes = align_up((size_t)n_q * n_r * 4, 256);
    const size_t table_bytes = align_up(fmh_compare_workspace(n_r), 256);
    int rc = ws.part.ensure(x_bytes + table_bytes + align_up((size_t)n_r, 256));
    if (rc) return rc;
    uint32_t* d_x = (uint32_t*)ws.part.p;
    void* d_table = (uint8_t*)ws.part.p + x_bytes;
    uint8_t* d_flags = (uint8_t*)d_table + table_bytes;
    {
        Prof pr(ctx, s, 3, 4);
        rc = launch_fmh_compare(d_qh, d_q_off, n_q, d_rh, d_r_off, n_r, 1, KMERML_FMH_CONTAINMENT, ctx->sm_count, d_table,
                                d_x, nullptr, nullptr, s);
        if (!rc) rc = launch_fmh_greedy_flag(d_x, n_q, n_r, threshold, d_flags, s);
    }
    if (rc) return rc;
    std::vector<uint8_t> flags(n_r);
    std::vector<uint64_t> r_off(n_r + 1);
    uint64_t q_total = 0;
    KM_CUDA(cudaMemcpyAsync(flags.data(), d_flags, (size_t)n_r, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaMemcpyAsync(r_off.data(), d_r_off, (size_t)(n_r + 1) * 8, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaMemcpyAsync(&q_total, d_q_off + n_q, 8, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    // the candidates: reference index | where its hashes begin | compact CSR offsets
    std::vector<int> cand;
    for (int r = 0; r < n_r; r++)
        if (flags[r]) cand.push_back(r);
    const int n_c = (int)cand.size();
    if (!n_c) return KMERML_OK;
    std::vector<uint64_t> index(2 * (size_t)n_c + 1);
    for (int c = 0; c < n_c; c++) {
        index[c] = r_off[cand[c]];
        index[n_c + c + 1] = index[n_c + c] + (r_off[cand[c] + 1] - r_off[cand[c]]);
    }
    const uint64_t c_total = index[2 * (size_t)n_c];
    if (d_qa && q_total > 0x7fffffffull)
        return fail(KMERML_ERR_RANGE, "fmh gather with abundances: more than 2^31 - 1 query hashes in one call");

    // ws.scratch: candidate hashes | index | candidate list | u | d | pick | remaining | s_len | s_off | scan temp |
    // assigned flags (one byte per query hash) | S_t (at most every query hash) | pick count, inconsistency flag
    // [| with abundances: S_t's abundances | the same sorted | the sort's temp storage]
    size_t at = 0;
    auto take = [&](size_t bytes) { const size_t a = at; at += align_up(bytes, 256); return a; };
    const size_t uq = (size_t)n_q * n_c * 4;
    const size_t temp_bytes = align_up(fmh_greedy_scan_temp_bytes(n_q), 256);
    const size_t at_ch = take(c_total * 8), at_index = take(index.size() * 8), at_cand = take((size_t)n_c * 4);
    const size_t at_u = take(uq), at_d = take(uq), at_pick = take((size_t)n_q * 4), at_remaining = take((size_t)n_q * 4);
    const size_t at_s_len = take((size_t)(n_q + 1) * 8), at_s_off = take((size_t)(n_q + 1) * 8), at_temp = take(temp_bytes);
    const size_t at_assigned = take(q_total), at_s = take(q_total * 8), at_cnt = take(8);
    const size_t med_temp = d_qa ? align_up(fmh_greedy_median_temp_bytes(n_q, (int)q_total), 256) : 0;
    const size_t at_sa = d_qa ? take(q_total * 4) : 0, at_ss = d_qa ? take(q_total * 4) : 0;
    const size_t at_med_temp = d_qa ? take(med_temp) : 0;
    if ((rc = ws.scratch.ensure(at))) return rc;
    uint8_t* base = (uint8_t*)ws.scratch.p;
    uint64_t* d_ch = (uint64_t*)(base + at_ch);
    uint64_t* d_index = (uint64_t*)(base + at_index);
    const uint64_t* d_c_off = d_index + n_c;
    int* d_cand = (int*)(base + at_cand);
    uint32_t* d_u = (uint32_t*)(base + at_u);
    uint32_t* d_d = (uint32_t*)(base + at_d);
    int* d_pick = (int*)(base + at_pick);
    uint32_t* d_remaining = (uint32_t*)(base + at_remaining);
    unsigned long long* d_s_len = (unsigned long long*)(base + at_s_len);
    unsigned long long* d_s_off = (unsigned long long*)(base + at_s_off);
    uint8_t* d_assigned = base + at_assigned;
    uint64_t* d_s = (uint64_t*)(base + at_s);
    unsigned int* d_cnt = (unsigned int*)(base + at_cnt);
    // a pinned word pair for the per-round read of d_cnt
    Tables t{ws};
    const size_t at_h = t.take(8);
    if ((rc = t.open())) return rc;
    unsigned int* h_cnt = t.host<unsigned int>(at_h);

    KM_CUDA(cudaMemcpyAsync(d_index, index.data(), index.size() * 8, cudaMemcpyHostToDevice, s));
    KM_CUDA(cudaMemcpyAsync(d_cand, cand.data(), (size_t)n_c * 4, cudaMemcpyHostToDevice, s));
    KM_CUDA(cudaMemsetAsync(d_pick, 0, (size_t)n_q * 4, s));
    KM_CUDA(cudaMemsetAsync(d_s_len, 0, (size_t)(n_q + 1) * 8, s));
    if (q_total) KM_CUDA(cudaMemsetAsync(d_assigned, 0, q_total, s));
    KM_CUDA(cudaMemsetAsync(d_cnt, 0, 8, s));
    {
        Prof pr(ctx, s, 3, 1);
        if ((rc = launch_fmh_gather(d_rh, d_index, d_c_off, n_c, c_total, d_ch, s))) return rc;
    }
    GatherAbund ab{d_qa, (uint32_t*)(base + at_sa), (unsigned long long*)d_uw, (unsigned long long*)d_usq, 0, max_matches};
    for (int round = 0; round < max_matches; round++) {
        KM_CUDA(cudaMemsetAsync(d_cnt, 0, 4, s));
        {
            Prof pr(ctx, s, 3, 1);
            rc = launch_fmh_greedy_select(d_u, d_d, n_c, d_x, n_q, n_r, d_cand, d_q_off, round, threshold, max_matches, d_pick,
                                          d_remaining, d_s_len, d_n_matches, d_ref, d_unique, d_inter, d_rem, d_cnt, s);
            if (rc) return rc;
        }
        KM_CUDA(cudaMemcpyAsync(h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, s));
        KM_CUDA(cudaStreamSynchronize(s));
        // the last round's remove assigned other counts than its select recorded: only unsorted or repeated input
        // values do that (a round always ends in a select, so every remove is checked)
        if (h_cnt[1]) return fail(KMERML_ERR_ARG, "fmh gather: the sketches must hold ascending, distinct values");
        const bool last = round + 1 == max_matches;
        if (!h_cnt[0] || (last && !d_qa)) break;
        Prof pr(ctx, s, 3, (d_qa ? 3 : 0) + (last ? 2 : 5));
        ab.round = round;
        rc = launch_fmh_greedy_remove(d_qh, d_q_off, n_q, d_ch, d_c_off, d_pick, d_s_len, d_s_off, base + at_temp,
                                      temp_bytes, d_assigned, d_s, d_cnt + 1, d_qa ? &ab : nullptr, s);
        if (!rc && d_qa)
            rc = launch_fmh_greedy_median(ab, d_s_off, d_pick, n_q, (int)q_total, (uint32_t*)(base + at_ss),
                                          base + at_med_temp, med_temp, d_med, s);
        if (rc) return rc;
        if (last) {                                   // no select follows: check this remove here
            KM_CUDA(cudaMemcpyAsync(h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, s));
            KM_CUDA(cudaStreamSynchronize(s));
            if (h_cnt[1]) return fail(KMERML_ERR_ARG, "fmh gather: the sketches must hold ascending, distinct values");
            break;
        }
        rc = launch_fmh_compare(d_s, (const uint64_t*)d_s_off, n_q, d_ch, d_c_off, n_c, 1, KMERML_FMH_CONTAINMENT,
                                ctx->sm_count, d_table, d_d, nullptr, nullptr, s);
        if (rc) return rc;
    }
    return KMERML_OK;
}

int kmerml_fmh_gather(kmerml_ctx* ctx, const uint64_t* d_q_hashes, const uint64_t* d_q_offsets, int n_q,
                      const uint64_t* d_r_hashes, const uint64_t* d_r_offsets, int n_r, uint32_t threshold, int max_matches,
                      int32_t* d_n_matches, int32_t* d_match_ref, uint32_t* d_match_unique, uint32_t* d_match_intersect,
                      uint32_t* d_match_remaining, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (threshold < 1) return fail(KMERML_ERR_ARG, "threshold must be >= 1");
    if (max_matches < 1) return fail(KMERML_ERR_ARG, "max_matches must be >= 1");
    if (n_q < 0 || n_r < 0) return fail(KMERML_ERR_ARG, "n_q and n_r must be >= 0");
    if (!n_q) return KMERML_OK;
    if (!d_q_offsets || !d_r_offsets || !d_n_matches || !d_match_ref || !d_match_unique || !d_match_intersect ||
        !d_match_remaining)
        return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return fmh_gather_core(ctx, d_q_hashes, d_q_offsets, n_q, d_r_hashes, d_r_offsets, n_r, threshold, max_matches,
                           d_n_matches, d_match_ref, d_match_unique, d_match_intersect, d_match_remaining, nullptr,
                           nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int kmerml_fmh_gather_abundance(kmerml_ctx* ctx, const uint64_t* d_q_hashes, const uint64_t* d_q_offsets, int n_q,
                                const uint64_t* d_r_hashes, const uint64_t* d_r_offsets, int n_r, uint32_t threshold,
                                int max_matches, int32_t* d_n_matches, int32_t* d_match_ref, uint32_t* d_match_unique,
                                uint32_t* d_match_intersect, uint32_t* d_match_remaining, const uint32_t* d_q_abundances,
                                uint64_t* d_match_unique_weighted, uint64_t* d_match_unique_sumsq,
                                double* d_match_median_abund, void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (threshold < 1) return fail(KMERML_ERR_ARG, "threshold must be >= 1");
    if (max_matches < 1) return fail(KMERML_ERR_ARG, "max_matches must be >= 1");
    if (n_q < 0 || n_r < 0) return fail(KMERML_ERR_ARG, "n_q and n_r must be >= 0");
    if (!n_q) return KMERML_OK;
    if (!d_q_offsets || !d_r_offsets || !d_n_matches || !d_match_ref || !d_match_unique || !d_match_intersect ||
        !d_match_remaining || !d_q_abundances || !d_match_unique_weighted || !d_match_unique_sumsq ||
        !d_match_median_abund)
        return fail(KMERML_ERR_ARG, "null pointer argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    return fmh_gather_core(ctx, d_q_hashes, d_q_offsets, n_q, d_r_hashes, d_r_offsets, n_r, threshold, max_matches,
                           d_n_matches, d_match_ref, d_match_unique, d_match_intersect, d_match_remaining, d_q_abundances,
                           d_match_unique_weighted, d_match_unique_sumsq, d_match_median_abund, (cudaStream_t)stream);
}

// NCCL through the process that called us (no link-time dependency): the four entry points the exchange needs.
namespace {
struct NcclApi {
    int (*all_reduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*reduce_scatter)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*comm_count)(void*, int*) = nullptr;
    int (*comm_user_rank)(void*, int*) = nullptr;
    const char* (*get_error_string)(int) = nullptr;
    bool ok = false;
};
const NcclApi& nccl_api() {
    static const NcclApi api = [] {
        NcclApi a;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);      // the copy that is already in the process
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return a;
        a.all_reduce = reinterpret_cast<decltype(a.all_reduce)>(dlsym(h, "ncclAllReduce"));
        a.reduce_scatter = reinterpret_cast<decltype(a.reduce_scatter)>(dlsym(h, "ncclReduceScatter"));
        a.comm_count = reinterpret_cast<decltype(a.comm_count)>(dlsym(h, "ncclCommCount"));
        a.comm_user_rank = reinterpret_cast<decltype(a.comm_user_rank)>(dlsym(h, "ncclCommUserRank"));
        a.get_error_string = reinterpret_cast<decltype(a.get_error_string)>(dlsym(h, "ncclGetErrorString"));
        a.ok = a.all_reduce && a.reduce_scatter && a.comm_count && a.comm_user_rank;
        return a;
    }();
    return api;
}
}  // namespace

int kmerml_allreduce_counts(kmerml_ctx* ctx, void* nccl_comm, void* d_counts, uint64_t n, int dtype, int reduce_scatter,
                            void* stream) {
    if (!ctx || !nccl_comm || (n && !d_counts)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (dtype < 0 || dtype > 1) return fail(KMERML_ERR_ARG, "dtype must be 0 (uint32) or 1 (uint64)");
    const NcclApi& nccl = nccl_api();
    if (!nccl.ok) return fail(KMERML_ERR_ARG, "no NCCL in this process (libnccl.so.2 could not be opened)");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    if (!n) return KMERML_OK;
    constexpr int NCCL_UINT32 = 3, NCCL_UINT64 = 5, NCCL_SUM = 0;      // ncclDataType_t / ncclRedOp_t (nccl.h)
    const int type = dtype == 0 ? NCCL_UINT32 : NCCL_UINT64;
    const size_t elem = dtype == 0 ? 4 : 8;
    auto nccl_fail = [&](int e, const char* what) {
        return fail(KMERML_ERR_CUDA, std::string(what) + ": " + (nccl.get_error_string ? nccl.get_error_string(e) : "NCCL error"));
    };
    int e;
    if (!reduce_scatter) {
        if ((e = nccl.all_reduce(d_counts, d_counts, (size_t)n, type, NCCL_SUM, nccl_comm, (cudaStream_t)stream)))
            return nccl_fail(e, "ncclAllReduce");
        return KMERML_OK;
    }
    int ranks = 0, rank = 0;
    if ((e = nccl.comm_count(nccl_comm, &ranks))) return nccl_fail(e, "ncclCommCount");
    if ((e = nccl.comm_user_rank(nccl_comm, &rank))) return nccl_fail(e, "ncclCommUserRank");
    if (ranks <= 0 || n % (uint64_t)ranks) return fail(KMERML_ERR_ARG, "the row length must be a multiple of the number of ranks");
    const size_t per = (size_t)(n / (uint64_t)ranks);
    if ((e = nccl.reduce_scatter(d_counts, (uint8_t*)d_counts + (size_t)rank * per * elem, per, type, NCCL_SUM, nccl_comm,
                                 (cudaStream_t)stream)))
        return nccl_fail(e, "ncclReduceScatter");
    return KMERML_OK;
}

int kmerml_encode(kmerml_ctx* ctx, const uint8_t* d_fasta, uint64_t nbytes, uint8_t* d_symbols, uint64_t* d_tallies,
                  void* stream) {
    if (!ctx) return fail(KMERML_ERR_ARG, "ctx is null");
    if (nbytes && (!d_fasta || !d_symbols)) return fail(KMERML_ERR_ARG, "null pointer argument");
    if (((uintptr_t)d_fasta & 15)) return fail(KMERML_ERR_ARG, "device pointers must be 16-byte aligned");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(KMERML_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t s = (cudaStream_t)stream;
    Workspace& ws = ctx->ws[0];
    if (int orc = order_stream(ctx, (cudaStream_t)stream)) return orc;
    if (d_tallies) {
        int rc = launch_genome_stats(d_fasta, nbytes, (unsigned long long*)d_tallies, s);
        if (rc) return rc;
        ctx->launches += 1;
    }
    if (!nbytes) return KMERML_OK;
    KM_CUDA(cudaMemsetAsync(d_symbols, 0xFF, (size_t)nbytes, s));
    DevWalk w;
    int rc = put_single_walk(ws, d_fasta, nbytes, atomic_slice_bytes(ctx->sm_count, nbytes), TILE_BYTES, s, &w);
    if (rc) return rc;
    ctx->launches += 1;
    return launch_encode(d_fasta, w.genomes, w.slices, w.n_slices, d_symbols, s);
}

}  // extern "C"
