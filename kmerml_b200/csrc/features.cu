// features.cu -- record table, genome tallies, static per-k-mer features, row normalisation and the
// genome x genome distance matrix.
//
// Reference points (paths relative to the reference tree):
//   scan_records      the per-record bookkeeping of kmerml/kmers/generate.py:39-46,60
//                     (record ids come from the header lines, "too short" from lengths)
//   genome_stats      contigs / total size / G+C / N of kmerml/utils/genome_metadata.py:55-85
//   static_features   kmerml/kmers/statistics.py:190-240 (_add_gc / _add_base_count /
//                     _add_presence / _add_cpg / _add_entropy / _add_repeat): every one
//                     of them is a function of the k-mer string only, so one table per k
//   normalize_rows    the normalize(method="frequency") the reference only gestures at
//                     (tests/test_ml.py:8)
//   pairwise          cosine / Euclidean distances the stubs in kmerml/ml/clustering.py
//                     would consume (SURVEY 8a row 13)
#include "fasta_walk.cuh"
#include "internal.h"

namespace km {

// ------------------------------------------------------------------ records
__global__ void find_headers_kernel(const uint8_t* __restrict__ buf, uint64_t lo, uint64_t hi,
                                    unsigned long long* offsets, uint32_t cap, uint32_t* count) {
    const uint64_t cs = lo + ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 64;
    if (cs >= hi) return;
    const uint64_t ce = cs + 64 < hi ? cs + 64 : hi;
    for (uint64_t p = cs; p < ce; p++) {
        if (buf[p] != (uint8_t)'>') continue;
        if (!(p == lo || is_term(buf[p - 1]))) continue;
        uint32_t slot = atomicAdd(count, 1u);
        if (slot < cap) offsets[slot] = p - lo;
    }
}

// One thread per record: does it hold fewer than `need` symbols?
__global__ void record_short_kernel(const uint8_t* __restrict__ buf, uint64_t lo, uint64_t hi,
                                    const unsigned long long* __restrict__ offsets, uint32_t n, int need,
                                    uint8_t* is_short) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Genome g;
    g.b = buf;
    g.lo = lo;
    g.hi = hi;
    uint64_t p = lo + offsets[i];
    while (p < hi && !is_term(buf[p])) p++;          // end of the header line
    int total = 0;
    uint64_t r = p;
    while (total < need) {
        if (next_symbol(g, r) == SYM_HDR) break;
        total++;
    }
    is_short[i] = total < need ? 1 : 0;
}

int launch_scan_records(const uint8_t* d_fasta, uint64_t nbytes, int need, unsigned long long* d_offsets,
                        uint8_t* d_short, uint32_t cap, uint32_t* d_count, cudaStream_t s) {
    KM_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint32_t), s));
    if (!nbytes) return KMERML_OK;
    // the first header line (text before it is ignored) is found by a single thread
    // inside find_headers_kernel's p == lo rule, so give it the true start:
    uint64_t threads = (nbytes + 63) / 64;
    find_headers_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(d_fasta, 0, nbytes, d_offsets, cap, d_count);
    KM_CUDA(cudaGetLastError());
    (void)need; (void)d_short;
    return KMERML_OK;
}

int launch_record_short(const uint8_t* d_fasta, uint64_t nbytes, const unsigned long long* d_offsets, uint32_t n,
                        int need, uint8_t* d_short, cudaStream_t s) {
    if (!n) return KMERML_OK;
    record_short_kernel<<<(n + 127) / 128, 128, 0, s>>>(d_fasta, 0, nbytes, d_offsets, n, need, d_short);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

// ----------------------------------------------------------- genome stats
// contigs / total_size / G+C / N tallies as kmerml/utils/genome_metadata.py:55-85 computes them
// (upper-cased sequence of every record; len(sequence) counts every symbol, valid base or not).
// out[0] contigs, out[1] total_size, out[2] gc_count, out[3] n_count.  One thread per 64-byte chunk.
// No thread needs to know whether its chunk starts inside a header line: every byte is tallied as if
// it were sequence, and the thread that meets a header start ('>' at a line start) walks that one line
// and takes its bytes' tallies back out.  The sums wrap mod 2^64, so the order does not matter.
__global__ void genome_stats_kernel(const uint8_t* __restrict__ buf, uint64_t nbytes, unsigned long long* out) {
    __shared__ uint64_t s_lo;
    if (threadIdx.x == 0) s_lo = first_header(buf, 0, nbytes);
    __syncthreads();
    Genome g;
    g.b = buf;
    g.lo = s_lo;
    g.hi = nbytes;
    const uint64_t cb = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 64;
    const uint64_t cs = cb > g.lo ? cb : g.lo;
    const uint64_t ce = cb + 64 < g.hi ? cb + 64 : g.hi;
    // 64-bit wrap-around arithmetic all the way (a warp's net tally can be negative when a header line
    // crosses its span: with 32-bit tallies zero-extended into the 64-bit sums that added 2^32)
    unsigned long long contigs = 0, total = 0, gc = 0, nn = 0;
    auto tally = [&](uint64_t pos, unsigned long long sign) -> bool {  // true: a header line starts at pos
        const uint32_t c = buf[pos];
        const int code = base_code(c);
        if (code >= 0) {
            total += sign;
            gc += (code == 1 || code == 2) ? sign : 0ull;
            return false;
        }
        const int kind = classify_nonbase(g, pos, c);
        if (kind == SYM_SKIP) return false;
        if (kind == SYM_HDR) return true;
        total += sign;
        nn += ((c & 0xDFu) == (uint32_t)'N') ? sign : 0ull;
        return false;
    };
    for (uint64_t pos = cs; pos < ce; pos++) {
        if (!tally(pos, 1ull)) continue;
        contigs++;
        for (uint64_t q = pos + 1; q < g.hi && !is_term(buf[q]); q++) tally(q, ~0ull);
    }
    // warp then global reduction
    for (int o = 16; o > 0; o >>= 1) {
        contigs += __shfl_xor_sync(0xffffffffu, contigs, o);
        total += __shfl_xor_sync(0xffffffffu, total, o);
        gc += __shfl_xor_sync(0xffffffffu, gc, o);
        nn += __shfl_xor_sync(0xffffffffu, nn, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (contigs) atomicAdd(out + 0, contigs);
        if (total) atomicAdd(out + 1, total);
        if (gc) atomicAdd(out + 2, gc);
        if (nn) atomicAdd(out + 3, nn);
    }
}

int launch_genome_stats(const uint8_t* d_fasta, uint64_t nbytes, unsigned long long* d_out, cudaStream_t s) {
    KM_CUDA(cudaMemsetAsync(d_out, 0, 4 * sizeof(unsigned long long), s));
    if (!nbytes) return KMERML_OK;
    const uint64_t threads = (nbytes + 63) / 64;
    genome_stats_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(d_fasta, nbytes, d_out);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

// --------------------------------------------------------- static features
// out[idx * 8 + f] (int32), idx = lexicographic ACGT index of the k-mer:
//   0 n (length of the string the features are computed on)   4 T_count
//   1 A_count   2 C_count   3 G_count                          5 cpg_count   6 has_repeat
//   7 first base code of the string (for callers that rebuild it)
// compat != 0 reproduces the reference's CSV quirk (SURVEY section 0): the digit string
// (A0 T1 C2 G3) is parsed as an integer, so leading 'A's are lost and all-A becomes "A".
__global__ void static_features_kernel(int k, int compat, int32_t* out) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_kmers = 1u << (2 * k);
    if (idx >= n_kmers) return;
    int start = 0;
    if (compat) {
        while (start < k - 1 && ((idx >> (2 * (k - 1 - start))) & 3u) == 0u) start++;
    }
    const int n = k - start;
    int cnt[4] = {0, 0, 0, 0};
    int cpg = 0, rep = 0;
    int prev = -1;
    for (int i = start; i < k; i++) {
        const int c = (idx >> (2 * (k - 1 - i))) & 3;
        cnt[c]++;
        if (prev == 1 && c == 2) cpg++;            // "CG"
        prev = c;
    }
    for (int i = start; i + 3 < k; i++) {
        const uint32_t d0 = (idx >> (2 * (k - 2 - i))) & 15u;     // s[i:i+2]
        const uint32_t d1 = (idx >> (2 * (k - 4 - i))) & 15u;     // s[i+2:i+4]
        if (d0 == d1) { rep = 1; break; }
    }
    int32_t* o = out + (size_t)idx * 8;
    o[0] = n;
    o[1] = cnt[0]; o[2] = cnt[1]; o[3] = cnt[2]; o[4] = cnt[3];
    o[5] = cpg;
    o[6] = rep;
    o[7] = (idx >> (2 * (k - 1 - start))) & 3;
}

int launch_static_features(int k, int compat, int32_t* d_out, cudaStream_t s) {
    const uint32_t n = 1u << (2 * k);
    static_features_kernel<<<(n + 255) / 256, 256, 0, s>>>(k, compat, d_out);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

// ------------------------------------------------------------ normalisation
__global__ void normalize_rows_kernel(const uint32_t* __restrict__ counts, uint64_t counts_stride,
                                      const uint64_t* __restrict__ totals, uint64_t m, float* out,
                                      uint64_t out_stride) {
    const uint64_t g = blockIdx.y;
    const unsigned long long t = totals[g];
    const double inv = t ? 1.0 / (double)t : 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x)
        out[g * out_stride + i] = (float)((double)counts[g * counts_stride + i] * inv);
}

int launch_normalize_rows(const uint32_t* d_counts, uint64_t counts_stride, const uint64_t* d_totals, int n_rows,
                          uint64_t m, float* d_out, uint64_t out_stride, cudaStream_t s) {
    if (n_rows <= 0 || !m) return KMERML_OK;
    unsigned gx = (unsigned)std::min<uint64_t>((m + 255) / 256, 148u * 8u);
    for (int r0 = 0; r0 < n_rows; r0 += 32768) {
        int nr = std::min(32768, n_rows - r0);
        normalize_rows_kernel<<<dim3(gx, nr), 256, 0, s>>>(d_counts + (size_t)r0 * counts_stride, counts_stride,
                                                             d_totals + r0, m, d_out + (size_t)r0 * out_stride, out_stride);
        KM_CUDA(cudaGetLastError());
    }
    return KMERML_OK;
}

// ---------------------------------------------------------------- distances
// Gram matrix G = X X^T in float64 (fp32 / uint32 rows are widened on load, products
// and sums are fp64: the 1e-6 relative tolerance of the north star needs more than an
// fp32 accumulator over 65536 terms).  64 x 64 output tile per CTA, 4 x 4 per thread,
// K tiled by 16 through shared memory.
template <class T>
__global__ void __launch_bounds__(256)
gram_kernel(const T* __restrict__ X, uint64_t stride, int n, uint64_t m, double* __restrict__ G) {
    __shared__ double As[16][64 + 1];
    __shared__ double Bs[16][64 + 1];
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj < bi) return;                               // symmetric: upper triangle only
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
    for (uint64_t k0 = 0; k0 < m; k0 += 16) {
        // 64 rows x 16 columns of each operand: 1024 elements, 4 per thread
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int lin = threadIdx.x + e * 256;
            const int r = lin >> 4, c = lin & 15;
            const int ra = bi * 64 + r, rb = bj * 64 + r;
            const uint64_t col = k0 + c;
            As[c][r] = (ra < n && col < m) ? (double)X[(uint64_t)ra * stride + col] : 0.0;
            Bs[c][r] = (rb < n && col < m) ? (double)X[(uint64_t)rb * stride + col] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; kk++) {
            double a[4], b[4];
#pragma unroll
            for (int q = 0; q < 4; q++) { a[q] = As[kk][ty * 4 + q]; b[q] = Bs[kk][tx * 4 + q]; }
#pragma unroll
            for (int p = 0; p < 4; p++)
#pragma unroll
                for (int q = 0; q < 4; q++) acc[p][q] = fma(a[p], b[q], acc[p][q]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int p = 0; p < 4; p++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int r = bi * 64 + ty * 4 + p, c = bj * 64 + tx * 4 + q;
            if (r < n && c < n) {
                G[(uint64_t)r * n + c] = acc[p][q];
                G[(uint64_t)c * n + r] = acc[p][q];
            }
        }
}

__global__ void distance_from_gram_kernel(const double* __restrict__ G, int n, int metric, float* D32, double* D64) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)n * n) return;
    const int i = (int)(idx / n), j = (int)(idx % n);
    const double d = i == j ? 0.0 : gram_distance(G[(uint64_t)i * n + i], G[(uint64_t)j * n + j], G[idx], metric);
    if (D32) D32[idx] = (float)d;
    if (D64) D64[idx] = d;
}

int launch_pairwise(const void* d_x, int dtype, uint64_t stride, int n, uint64_t m, int metric, double* d_gram,
                    float* d_out32, double* d_out64, cudaStream_t s) {
    if (n <= 0) return KMERML_OK;
    const unsigned nb = (unsigned)((n + 63) / 64);
    if (dtype == 0) gram_kernel<float><<<dim3(nb, nb), 256, 0, s>>>((const float*)d_x, stride, n, m, d_gram);
    else if (dtype == 1) gram_kernel<uint32_t><<<dim3(nb, nb), 256, 0, s>>>((const uint32_t*)d_x, stride, n, m, d_gram);
    else gram_kernel<double><<<dim3(nb, nb), 256, 0, s>>>((const double*)d_x, stride, n, m, d_gram);
    KM_CUDA(cudaGetLastError());
    const uint64_t nn = (uint64_t)n * n;
    distance_from_gram_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, s>>>(d_gram, n, metric, d_out32, d_out64);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

}  // namespace km
