// sparse_walk.cuh -- the 64-bit k-mer walker of the sparse path (k <= 32), shared by sparse_emit_kernel (sparse.cu:
// every window) and sketch_emit_kernel (sketch.cu: the windows whose hash is at most a threshold).  The FASTA window
// rules live here once; a kernel supplies only the sink that receives the canonical key of every window.
#pragma once
#include "fasta_walk.cuh"
#include "internal.h"

namespace km {

struct SparseParams {
    int k;
    int min_rec;
    int canonical;
    uint64_t mask;       // 4^k - 1 (all ones for k = 32)
};

constexpr int SPARSE_THREADS = 256;
constexpr int SPARSE_TILE = SPARSE_THREADS * CHUNK;          // 8 KB
constexpr int SPARSE_TILES_PER_SLICE = 16;                   // one CTA walks 128 KB
static_assert(SPARSE_TILE == SPARSE_TILE_BYTES && SPARSE_TILE * SPARSE_TILES_PER_SLICE == SPARSE_SLICE_BYTES,
              "internal.h states the sparse walker's tile and slice sizes for the host");

// A sink takes the windows of one CTA's slice:
//   lanes = fast_begin(fast, fast_mask, n31_mask, lane)  every lane of a warp that has fast lanes, before their windows
//   fast_window(lanes, j, key, pos)                     window j (0..31) of a fast lane's clean chunk
//   window(key, pos)                                    a window of the byte walker (any subset of the warp's lanes)
// pos is the byte offset of the window's last base.
//
// One thread per 32-byte chunk, owning the windows whose last base lies in it.
//   * Clean chunk (only bases and at most one '\n') after a clean chunk -- nearly every chunk of a wrapped
//     genome: two 128-bit loads, the SWAR classifier and bit-compaction of fasta_walk.cuh, the k-1 bases before
//     the chunk from the neighbour thread's packed chunk (31 or 32 bases: enough for k <= 32) through shared
//     memory, then a rolling 64-bit forward k-mer and reverse complement, one shift-or each per base.
//   * Anything else (header lines, N runs, IUPAC, '\r', the first chunk of a slice ...): the byte walker whose
//     start state comes from a backward walk over global memory (same rules as the dense generic path).
// Whether a chunk starts inside a header line is settled per tile: the slice table says so for the slice's
// first byte, and header lines that start inside the tile flag the chunks they cover.
template <class Sink>
__device__ __forceinline__ void walk_sparse_slice(const uint8_t* __restrict__ buf, const GenomeDev& gd, const Slice& sl,
                                                  const SparseParams& P, const Sink& sink) {
    __shared__ uint8_t s_flags[SPARSE_THREADS];
    __shared__ unsigned long long s_carry[2];
    __shared__ uint2 s_packed[SPARSE_THREADS];              // the chunk's bases, top-aligned (hi, lo) ...
    __shared__ uint8_t s_n[SPARSE_THREADS];                 // ... and how many: 31 / 32, 0 = not a clean chunk
    __shared__ uint2 s_prev_packed;                          // the last chunk of the tile before
    __shared__ uint32_t s_prev_n;
    const int tid = threadIdx.x, lane = tid & 31;
    Genome g;
    g.b = buf;
    g.lo = gd.lo;
    g.hi = gd.hi;
    if (tid == 0) { s_carry[0] = s_carry[1] = sl.hdr_until; s_prev_n = 0; s_prev_packed = make_uint2(0, 0); }
    const int rcshift = 2 * (P.k - 1);
    const uint64_t end = sl.end < g.hi ? sl.end : g.hi;
    for (uint64_t tb = sl.begin; tb < end; tb += SPARSE_TILE) {
        s_flags[tid] = 0;
        __syncthreads();
        const uint64_t cb = tb + (uint64_t)tid * CHUNK;
        const uint64_t cs = cb > g.lo ? cb : g.lo;
        const uint64_t ce = cb + CHUNK < g.hi ? cb + CHUNK : g.hi;
        const bool has = cs < ce;
        CleanChunk cc;
        cc.hi = cc.lo = 0; cc.n = 0; cc.nl = 32; cc.last16 = 0;
        bool clean = false;
        auto on_header = [&](uint64_t, uint64_t until) {
            for (int j = tid + 1; j < SPARSE_THREADS && tb + (uint64_t)j * CHUNK < until; j++) s_flags[j] = 1;
            atomicMax(&s_carry[1], (unsigned long long)until);
        };
        if (has && cb >= g.lo && cb + CHUNK <= g.hi) {
            uint32_t w[CHUNK / 4];
            const uint4* src = reinterpret_cast<const uint4*>(buf + cb);
#pragma unroll
            for (int i = 0; i < CHUNK / 16; i++) {
                const uint4 v = __ldg(src + i);
                w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
            }
            clean = classify_pack(w, cc);
            if (!clean && any_byte_eq_chunk(w, 0x3E3E3E3Eu)) find_headers(g, cs, ce, on_header);
        } else if (has) {
            find_headers(g, cs, ce, on_header);
        }
        s_packed[tid] = make_uint2(cc.hi, cc.lo);
        s_n[tid] = clean ? (uint8_t)cc.n : 0;
        __syncthreads();
        int in_hdr = (s_flags[tid] || cs < s_carry[0]) ? 1 : 0;
        const bool starts_in_hdr = in_hdr != 0;
        // the chunk before: clean, in sequence, not shadowed by a header line
        uint2 pv;
        uint32_t pn;
        if (tid > 0) {
            pv = s_packed[tid - 1];
            pn = (s_flags[tid - 1] || (cb - CHUNK) < s_carry[0]) ? 0u : s_n[tid - 1];
        } else {
            pv = s_prev_packed;
            pn = s_prev_n;
        }
        const bool fast = has && clean && !in_hdr && pn != 0 && P.min_rec <= P.k;
        // ---- fast lanes
        const unsigned fast_mask = __ballot_sync(0xffffffffu, fast);
        if (fast_mask) {
            const unsigned n31_mask = __ballot_sync(0xffffffffu, fast && cc.n == 31);
            const auto lanes = sink.fast_begin(fast, fast_mask, n31_mask, lane);
            if (fast) {
                // the k-1 bases before the chunk: the last ones of the neighbour's pn bases
                const uint64_t prev = (((uint64_t)pv.x << 32) | pv.y) >> (64 - 2 * pn);
                uint64_t fwd = prev & (P.mask >> 2);
                uint64_t rc = 0;
                for (int i = P.k - 2; i >= 0; i--)                   // oldest first
                    rc = (rc >> 2) | ((uint64_t)(3u - (uint32_t)((prev >> (2 * i)) & 3u)) << rcshift);
                const uint64_t own = ((uint64_t)cc.hi << 32) | cc.lo;
#pragma unroll 4
                for (int j = 0; j < 32; j++) {
                    if (j >= cc.n) break;
                    const uint32_t code = (uint32_t)(own >> (62 - 2 * j)) & 3u;
                    fwd = ((fwd << 2) | code) & P.mask;
                    rc = (rc >> 2) | ((uint64_t)(3u - code) << rcshift);
                    sink.fast_window(lanes, j, P.canonical ? (fwd < rc ? fwd : rc) : fwd,
                                     cs + (uint64_t)(j + (j >= cc.nl ? 1 : 0)));
                }
            }
        }
        // ---- everything else: the byte walker
        if (has && !fast) {
            uint64_t fwd = 0, rc = 0;
            int run = 0, rec_known = 0;
            if (!in_hdr && cs > g.lo) {
                // the up to k-1 valid bases right before the chunk, oldest first
                uint64_t q = cs;
                uint32_t codes[32];
                int cnt = 0;
                while (cnt < P.k - 1) {
                    int kind = prev_symbol(g, q);
                    if (kind > 3) break;
                    codes[cnt++] = (uint32_t)kind;
                }
                for (int i = cnt - 1; i >= 0; i--) {
                    fwd = ((fwd << 2) | codes[i]) & P.mask;
                    rc = (rc >> 2) | ((uint64_t)(3u - codes[i]) << rcshift);
                }
                run = cnt;
            }
            for (uint64_t pos = cs; pos < ce; pos++) {
                const uint32_t c = buf[pos];
                const int code = base_code(c);
                if (code >= 0 && !in_hdr) {
                    fwd = ((fwd << 2) | (uint64_t)code) & P.mask;
                    rc = (rc >> 2) | ((uint64_t)(3 - code) << rcshift);
                    run++;
                    if (run >= P.k) {
                        if (P.min_rec > P.k) {
                            if (rec_known == 0) rec_known = (run >= P.min_rec || record_len_at_least(g, pos, P.min_rec)) ? 1 : 2;
                            if (rec_known == 2) continue;
                        }
                        sink.window(P.canonical ? (fwd < rc ? fwd : rc) : fwd, pos);
                    }
                    continue;
                }
                if (in_hdr) {
                    if (is_term(c)) in_hdr = 0;
                    continue;
                }
                const int kind = classify_nonbase(g, pos, c);
                if (kind == SYM_SKIP) continue;
                run = 0;
                fwd = rc = 0;
                if (kind == SYM_HDR) { in_hdr = 1; rec_known = 0; }
            }
        }
        __syncthreads();
        if (tid == 0) s_carry[0] = s_carry[1];
        if (tid == SPARSE_THREADS - 1) {
            const bool ok = has && clean && !starts_in_hdr;
            s_prev_packed = make_uint2(cc.hi, cc.lo);
            s_prev_n = ok ? (uint32_t)cc.n : 0u;
        }
    }
}

}  // namespace km
