// gram_tc.cu -- exact integer Gram matrix of count rows on the 5th-generation tensor cores.
//
// The genome x genome distance matrix (SURVEY 8a row 13) is the only dense contraction of the
// path.  The 1e-6 relative tolerance on 1 - cos(x, y) rules out bf16/tf32 products and an fp32
// accumulator over 65 536 terms, but the feature rows ARE integer counts, so the Gram matrix
//      G = C C^T,   C = sum_d 256^d D_d   (D_d = d-th byte of every count, uint8)
// is computed EXACTLY as   G = sum_{a,b} 256^(a+b) D_a D_b^T   with
//      tcgen05.mma.cta_group::1.kind::i8   (u8 x u8 -> s32 accumulators in TMEM),
// at most 8192 features per accumulation (255*255*8192 < 2^31; rows longer than 65535 * 8192 take up to 32768, the
// most that stays below 2^31), then summed in int64.
//
// One CTA (128 threads) owns a 128 x 128 tile of one (a, b) digit pair and one K split:
//   global uint8 rows --16 B loads--> registers --> shared memory in the UMMA canonical K-major,
//   no-swizzle core-matrix layout (8 rows x 16 B per core matrix) --> two MMAs (K = 32 each) per
//   64-byte K block, issued by one thread, tracked by an mbarrier (tcgen05.commit); the next
//   block's global loads are in flight while the tensor core works.  Epilogue: tcgen05.ld
//   (32 lanes x 32 columns per warp) and int64 atomicAdd of 256^(a+b) * acc into G.
//
// One launcher, launch_gram_planes, computes rows [row_begin, row_end) of G from the planes, all digit
// pairs in one launch where gridDim.z allows; over all n rows it runs only the tiles on or above the
// diagonal and mirrors each entry.  Every distance of count rows -- the whole matrix, a row block of
// uint32 rows, a row block of gathered planes -- is that Gram, then distance_rows_kernel on G and the
// exact squared norms.
#include "internal.h"

namespace km {

constexpr int GT_M = 128, GT_N = 128, GT_KB = 64;       // tile and K block (bytes = uint8 elements)
constexpr int GT_KSPLIT = 8192;                         // features per accumulation: 255^2 * 8192 < 2^31
constexpr int GT_KSPLIT_MAX = 32768;                    // ... and the most it can be: 255^2 * 32768 < 2^31
constexpr uint64_t GT_MAX_SPLITS = 65535;               // the K splits run along gridDim.z
constexpr int GT_THREADS = 128;

// The shortest K range per CTA (a multiple of GT_KB) that covers a row of m features in at most GT_MAX_SPLITS splits.
static uint64_t min_ksplit(uint64_t m) { return ((m + GT_MAX_SPLITS - 1) / GT_MAX_SPLITS + GT_KB - 1) / GT_KB * GT_KB; }

static int ksplit_out_of_range(uint64_t m) {
    set_error("count rows of " + std::to_string(m) + " features are longer than the Gram kernel's grid covers (" +
              std::to_string(GT_MAX_SPLITS * GT_KSPLIT_MAX) + ")");
    return KMERML_ERR_RANGE;
}

// One CTA per count row: its four byte planes (128-bit loads, one packed 32-bit store per plane and four bins), its
// exact squared norm (uint64, then double -- the Gram diagonal a row-block distance needs for ALL genomes) and the
// largest count (how many planes the Gram needs).  This is also what one rank of a sharded job runs on ITS rows
// before the planes -- not the uint32 rows -- are gathered (kmerml_count_planes).
__global__ void __launch_bounds__(256)
split_planes_kernel(const uint32_t* __restrict__ counts, uint64_t stride, uint64_t m, uint8_t* __restrict__ planes,
                    uint64_t plane_stride, double* __restrict__ sumsq, unsigned int* __restrict__ max_count) {
    const uint32_t row = blockIdx.x;
    const uint32_t* c = counts + (uint64_t)row * stride;
    uint8_t* out = planes + (uint64_t)row * m;
    unsigned long long acc = 0;
    unsigned int mx = 0;
    const bool vec = (reinterpret_cast<uintptr_t>(c) & 15) == 0 && ((reinterpret_cast<uintptr_t>(out) | plane_stride) & 3) == 0;
    if (vec) {
        for (uint64_t i = (uint64_t)threadIdx.x * 4; i < m; i += 256 * 4) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(c + i));
            mx = max(max(mx, v.x), max(max(v.y, v.z), v.w));
            acc += (unsigned long long)v.x * v.x + (unsigned long long)v.y * v.y + (unsigned long long)v.z * v.z +
                   (unsigned long long)v.w * v.w;
            // byte d of the four counts -> one word of plane d  (lo01 = x0 y0 x1 y1, hi01 = x2 y2 x3 y3, ...)
            const uint32_t lo01 = __byte_perm(v.x, v.y, 0x5140), hi01 = __byte_perm(v.x, v.y, 0x7362);
            const uint32_t lo23 = __byte_perm(v.z, v.w, 0x5140), hi23 = __byte_perm(v.z, v.w, 0x7362);
            *reinterpret_cast<uint32_t*>(out + i) = __byte_perm(lo01, lo23, 0x5410);
            *reinterpret_cast<uint32_t*>(out + plane_stride + i) = __byte_perm(lo01, lo23, 0x7632);
            *reinterpret_cast<uint32_t*>(out + 2 * plane_stride + i) = __byte_perm(hi01, hi23, 0x5410);
            *reinterpret_cast<uint32_t*>(out + 3 * plane_stride + i) = __byte_perm(hi01, hi23, 0x7632);
        }
    } else {
        for (uint64_t i = threadIdx.x; i < m; i += 256) {
            const uint32_t v = c[i];
            mx = max(mx, v);
            acc += (unsigned long long)v * v;
            out[i] = (uint8_t)v;
            out[plane_stride + i] = (uint8_t)(v >> 8);
            out[2 * plane_stride + i] = (uint8_t)(v >> 16);
            out[3 * plane_stride + i] = (uint8_t)(v >> 24);
        }
    }
    __shared__ unsigned long long s_acc[8];
    __shared__ unsigned int s_mx[8];
    for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0) { s_acc[threadIdx.x >> 5] = acc; s_mx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) { acc += s_acc[w]; mx = max(mx, s_mx[w]); }
        if (sumsq) sumsq[row] = (double)acc;
        if (mx) atomicMax(max_count, mx);
    }
}

int launch_count_planes(const uint32_t* d_counts, uint64_t stride, int n, uint64_t m, uint8_t* d_planes,
                        uint64_t plane_stride, double* d_sumsq, unsigned int* d_max, cudaStream_t s) {
    if (n <= 0) return KMERML_OK;
    split_planes_kernel<<<(unsigned)n, 256, 0, s>>>(d_counts, stride, m, d_planes, plane_stride, d_sumsq, d_max);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}


__device__ __forceinline__ uint64_t umma_desc_kmajor_noswizzle(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // cute::UMMA::SmemDescriptor: start >> 4 [0,14) | LBO >> 4 [16,30) | SBO >> 4 [32,46) | version 1 [46,48) | layout 0
    const uint32_t lo = ((smem_addr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
    const uint32_t hi = ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14);
    return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}

__global__ void __launch_bounds__(GT_THREADS)
gram_i8_kernel(const uint8_t* __restrict__ planes, uint64_t plane_stride, int n_planes, int n, uint64_t m,
               int row_tile0, int symmetric, uint32_t ksplit, uint32_t launch_pairs, uint32_t pair0,
               unsigned long long* __restrict__ G) {
    // Row block (symmetric = 0): tile rows row_tile0 .. row_tile0 + gridDim.y - 1 against all columns, G holds those
    // rows at their global row index.  Symmetric: every row, tiles on or above the diagonal only; entry (i, j >= i) is
    // added at (i, j) and, for j != i, at (j, i).
    // shared: A tile and B tile in core-matrix layout: [kg (4)][mg (16)][8 rows][16 B]
    __shared__ __align__(128) uint8_t sA[GT_M * GT_KB];
    __shared__ __align__(128) uint8_t sB[GT_N * GT_KB];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row0 = (blockIdx.y + row_tile0) * GT_M, col0 = blockIdx.x * GT_N;
    if (symmetric && col0 < row0) return;
    // digit pairs pair0 .. pair0 + launch_pairs - 1 in one launch: blockIdx.z = (pair - pair0) * splits + split
    const uint32_t splits = gridDim.z / launch_pairs;
    const uint32_t pair = pair0 + blockIdx.z / splits;
    const uint32_t a = pair / (uint32_t)n_planes, b = pair % (uint32_t)n_planes;
    const uint8_t* A = planes + (uint64_t)a * plane_stride;
    const uint8_t* B = planes + (uint64_t)b * plane_stride;
    const unsigned long long scale = 1ull << (8 * (a + b));  // n_planes <= 4: at most 2^48
    const uint64_t k_begin = (uint64_t)(blockIdx.z % splits) * ksplit;
    const uint64_t k_end = min(m, k_begin + ksplit);
    if (k_begin >= k_end) return;

    const uint32_t bar_addr = (uint32_t)__cvta_generic_to_shared(&bar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {                                        // 128 TMEM columns: the 128 x 128 s32 accumulator
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(
            (uint32_t)__cvta_generic_to_shared(&tmem_base_s)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_acc = tmem_base_s;

    const uint32_t sA_addr = (uint32_t)__cvta_generic_to_shared(sA);
    const uint32_t sB_addr = (uint32_t)__cvta_generic_to_shared(sB);
    // instruction descriptor (cute::UMMA::InstrDescriptor): c_format S32 = 2 [4,6), a/b format u8 = 0,
    // a/b K-major = 0, n_dim = N >> 3 [17,23), m_dim = M >> 4 [24,29)
    const uint32_t idesc = (2u << 4) | ((uint32_t)(GT_N >> 3) << 17) | ((uint32_t)(GT_M >> 4) << 24);

    // each thread moves 4 + 4 16-byte pieces per K block: piece q -> row q / 4, 16-byte column q % 4.  The source
    // pointers advance by one K block per load: computed from row * m instead, ptxas re-derives every address from the
    // kernel parameters in each block, which lengthens the loop by a half.
    uint4 ra[4], rb[4];
    const uint8_t* srcA[4];
    const uint8_t* srcB[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int q = tid + GT_THREADS * i, r = q >> 2, p = q & 3;
        srcA[i] = A + (uint64_t)(row0 + r) * m + k_begin + 16 * p;
        srcB[i] = B + (uint64_t)(col0 + r) * m + k_begin + 16 * p;
    }
    auto load_block = [&](uint64_t k0) {                    // called for k0 = k_begin, k_begin + GT_KB, ...
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int q = tid + GT_THREADS * i, r = q >> 2, p = q & 3;
            const bool kin = k0 + 16 * p < k_end;
            ra[i] = (row0 + r < n && kin) ? *reinterpret_cast<const uint4*>(srcA[i]) : make_uint4(0, 0, 0, 0);
            rb[i] = (col0 + r < n && kin) ? *reinterpret_cast<const uint4*>(srcB[i]) : make_uint4(0, 0, 0, 0);
            srcA[i] += GT_KB;
            srcB[i] += GT_KB;
        }
    };
    auto store_block = [&]() {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int q = tid + GT_THREADS * i, r = q >> 2, p = q & 3;
            const uint32_t off = (uint32_t)((p * 16 + (r >> 3)) * 128 + (r & 7) * 16);
            *reinterpret_cast<uint4*>(sA + off) = ra[i];
            *reinterpret_cast<uint4*>(sB + off) = rb[i];
        }
    };

    uint32_t phase = 0;
    bool first = true;
    load_block(k_begin);
    for (uint64_t k0 = k_begin; k0 < k_end; k0 += GT_KB) {
        if (!first) { mbar_wait(bar_addr, phase); phase ^= 1; }   // previous MMAs have consumed the tiles
        store_block();
        if (k0 + GT_KB < k_end) load_block(k0 + GT_KB);           // next block in flight during the MMAs
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> async proxy
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int j = 0; j < GT_KB / 32; j++) {
                // MMA j reads K bytes [32 j, 32 j + 32): core-matrix columns 2j and 2j+1
                const uint64_t da = umma_desc_kmajor_noswizzle(sA_addr + (uint32_t)(2 * j) * 16 * 128, 16 * 128, 128);
                const uint64_t db = umma_desc_kmajor_noswizzle(sB_addr + (uint32_t)(2 * j) * 16 * 128, 16 * 128, 128);
                const uint32_t accumulate = (first && j == 0) ? 0u : 1u;
                asm volatile(
                    "{\n\t"
                    ".reg .pred p;\n\t"
                    "setp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
                    "}\n" ::"r"(tmem_acc), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
                    : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_addr) : "memory");
        }
        first = false;
    }
    mbar_wait(bar_addr, phase);                              // the last MMAs are done
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // epilogue: warp w owns TMEM lanes (= tile rows) 32 w .. 32 w + 31
    const int gi = row0 + warp * 32 + lane;
#pragma unroll 1
    for (int c0 = 0; c0 < GT_N; c0 += 32) {
        uint32_t v[32];
        const uint32_t taddr = tmem_acc + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
              "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
              "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
              "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (gi < n) {
#pragma unroll
            for (int c = 0; c < 32; c++) {
                const int gj = col0 + c0 + c;
                if (gj >= n || !v[c] || (symmetric && gj < gi)) continue;
                const unsigned long long add = (unsigned long long)v[c] * scale;
                atomicAdd(G + (uint64_t)gi * n + gj, add);
                if (symmetric && gj != gi) atomicAdd(G + (uint64_t)gj * n + gi, add);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem_acc));
}

// Rows [row_begin, row_end) of the exact Gram matrix G (n x n, uint64) of the count rows whose n_planes (1..4) byte
// planes start at planes (plane d at planes + d * plane_stride, n x m bytes, m a multiple of 64).  G holds the rows of
// the touched tiles, at their global row index.  Over all n rows the launch is symmetric: only tiles with col0 >= row0,
// for all n_planes^2 ordered digit pairs -- the upper triangle of sum_{a,b} 256^(a+b) D_a D_b^T is that of G -- and
// each entry (i, j > i) is mirrored to (j, i).
int launch_gram_planes(const uint8_t* planes, uint64_t plane_stride, int n_planes, int n, uint64_t m, int row_begin,
                       int row_end, unsigned long long* G, cudaStream_t s) {
    if (min_ksplit(m) > (uint64_t)GT_KSPLIT_MAX) return ksplit_out_of_range(m);
    const bool symmetric = row_begin == 0 && row_end == n;
    const int t0 = row_begin / GT_M, t1 = (row_end + GT_M - 1) / GT_M;
    KM_CUDA(cudaMemsetAsync(G + (size_t)t0 * GT_M * n, 0, (size_t)(std::min(t1 * GT_M, n) - t0 * GT_M) * n * 8, s));
    // the K range of a CTA shrinks (down to 1024 features) until the tiles that do work, over all digit pairs, make
    // about four CTAs per SM: a row block of one rank of eight is 8 x 1 tiles, which at 8192 features per CTA and one
    // launch per pair left 64 CTAs at a time on 148 SMs
    const unsigned tiles = (unsigned)((n + GT_N - 1) / GT_N);
    const unsigned pairs = (unsigned)(n_planes * n_planes);
    const uint64_t live_tiles = symmetric ? (uint64_t)tiles * (tiles + 1) / 2 : (uint64_t)tiles * (unsigned)(t1 - t0);
    const uint64_t want_ctas = 148ull * 4;
    const uint64_t base = live_tiles * pairs;
    uint64_t splits = std::max<uint64_t>((m + GT_KSPLIT - 1) / GT_KSPLIT, (want_ctas + base - 1) / base);
    splits = std::min<uint64_t>(splits, std::max<uint64_t>(m / 1024, 1));
    uint64_t ksplit = ((m + splits - 1) / splits + GT_KB - 1) / GT_KB * GT_KB;
    ksplit = std::max<uint64_t>(std::min<uint64_t>(ksplit, GT_KSPLIT), min_ksplit(m));
    const unsigned ksplits = (unsigned)((m + ksplit - 1) / ksplit);
    // all digit pairs in one launch while K splits x pairs fit gridDim.z; otherwise (rows of k = 13 and 14) one
    // launch per pair
    const unsigned pairs_per_launch = (uint64_t)ksplits * pairs <= GT_MAX_SPLITS ? pairs : 1;
    for (unsigned p0 = 0; p0 < pairs; p0 += pairs_per_launch) {
        gram_i8_kernel<<<dim3(tiles, (unsigned)(t1 - t0), ksplits * pairs_per_launch), GT_THREADS, 0, s>>>(
            planes, plane_stride, n_planes, n, m, t0, symmetric ? 1 : 0, (uint32_t)ksplit, pairs_per_launch, p0, G);
        KM_CUDA(cudaGetLastError());
    }
    return KMERML_OK;
}

// rows [row_begin, row_end) of the distance matrix from the row block of G and the squared norms of all rows
__global__ void distance_rows_kernel(const unsigned long long* __restrict__ G, const double* __restrict__ norm2, int n,
                                     int row_begin, int row_end, int metric, float* D32, double* D64) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)(row_end - row_begin) * n) return;
    const int i = row_begin + (int)(idx / n), j = (int)(idx % n);
    const double d = i == j ? 0.0 : gram_distance(norm2[i], norm2[j], (double)G[(uint64_t)i * n + j], metric);
    if (D32) D32[idx] = (float)d;
    if (D64) D64[idx] = d;
}

static size_t round256(size_t bytes) { return (bytes + 255) / 256 * 256; }

// Workspace of the distance rows: the uint64 Gram matrix, then the squared norms, the largest count and the byte planes
// of n uint32 count rows of m features (m = 0 when the caller brings planes and norms).
size_t distance_rows_workspace(int n, uint64_t m) {
    return round256((size_t)n * n * 8) + round256((size_t)n * 8 + 8) + (size_t)4 * n * m;
}

// Rows [row_begin, row_end) of the n x n distance matrix from the byte planes of ALL n count rows (plane d at
// d_planes + d * plane_stride, n x m bytes) and their squared norms: also the unit one rank computes when the genomes
// were counted on several GPUs (SURVEY 8e, C3).  The Gram entries are exact (tcgen05 kind::i8), so the block is
// bit-identical to the same rows of the whole matrix.
int launch_distance_rows_planes(const uint8_t* d_planes, uint64_t plane_stride, int n_planes, int n, uint64_t m,
                                const double* d_sumsq, int row_begin, int row_end, int metric, void* workspace,
                                float* d_out32, double* d_out64, cudaStream_t s) {
    if (row_begin >= row_end) return KMERML_OK;
    unsigned long long* G = (unsigned long long*)workspace;
    if (int rc = launch_gram_planes(d_planes, plane_stride, n_planes, n, m, row_begin, row_end, G, s)) return rc;
    const uint64_t cells = (uint64_t)(row_end - row_begin) * n;
    distance_rows_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, s>>>(G, d_sumsq, n, row_begin, row_end, metric, d_out32, d_out64);
    KM_CUDA(cudaGetLastError());
    return KMERML_OK;
}

int planes_needed(unsigned int max_count) {
    return max_count >= (1u << 24) ? 4 : max_count >= (1u << 16) ? 3 : max_count >= (1u << 8) ? 2 : 1;
}

// The same from uint32 count rows resident on this GPU: planes + norms + largest count in one pass, then the above.
int launch_distance_rows_tc(const uint32_t* d_counts, uint64_t stride, int n, uint64_t m, int row_begin, int row_end,
                            int metric, void* workspace, float* d_out32, double* d_out64, cudaStream_t s) {
    if (row_begin >= row_end) return KMERML_OK;
    double* d_norm = (double*)((uint8_t*)workspace + round256((size_t)n * n * 8));
    unsigned int* d_max = (unsigned int*)(d_norm + n);
    uint8_t* planes = (uint8_t*)d_norm + round256((size_t)n * 8 + 8);
    const size_t plane = (size_t)n * m;
    KM_CUDA(cudaMemsetAsync(d_max, 0, 8, s));
    if (int rc = launch_count_planes(d_counts, stride, n, m, planes, plane, d_norm, d_max, s)) return rc;
    unsigned int h_max = 0;
    KM_CUDA(cudaMemcpyAsync(&h_max, d_max, 4, cudaMemcpyDeviceToHost, s));
    KM_CUDA(cudaStreamSynchronize(s));
    return launch_distance_rows_planes(planes, plane, planes_needed(h_max), n, m, d_norm, row_begin, row_end, metric,
                                       workspace, d_out32, d_out64, s);
}

}  // namespace km
