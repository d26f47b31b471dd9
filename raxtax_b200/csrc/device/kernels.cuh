// kernels.cuh -- hand-written sm_100a kernels of the raxtax query-classification path.
//
//   K0 build_bitrows_kernel    CSR postings (Tree.k_mer_map, tree.rs:41,134-137) -> bit rows in HBM
//   K1 kmers_kernel            2-bit packing + unique sorted 8-mers per query (utils.rs:17-40)
//   K2 hitcount_bitrows_kernel per-query hit counts (raxtax.rs:58-64) by positional popcount over bit rows,
//                              fused count histogram (prob.rs:13-19)
//   K2' fixup_exact_kernel     --skip-exact-matches zeroing (raxtax.rs:65-68) applied to counts + histogram
//   K3 prob_table_kernel       highest-hit probabilities (prob.rs:20-102) on the windows that can matter
//   K4 prefix_kernel           prefix sums of the probabilities at node boundaries (lineage.rs:61-77,114-117)
//   K5 lineage_walk_kernel     tree walk with the 0.01 cutoff / fallback (lineage.rs:119-179), signals and ordering
//                              (lineage.rs:86-111), override (raxtax.rs:73-84)
//      best_hits_kernel        optional: each query's T references with the most shared 8-mers, from the resident count row
#pragma once

#include <math_constants.h>

#include "common.cuh"

namespace rtx {

// =========================================================================================================
// small helpers
// =========================================================================================================
__device__ __forceinline__ uint2 ldg_stream(const uint2* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

// inclusive warp scan
__device__ __forceinline__ double warp_scan_incl(double v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        double y = __shfl_up_sync(kFullMask, v, o);
        if (lane >= o) v += y;
    }
    return v;
}
__device__ __forceinline__ u32 warp_scan_incl(u32 v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 y = __shfl_up_sync(kFullMask, v, o);
        if (lane >= o) v += y;
    }
    return v;
}

// Deterministic block-wide sum, result broadcast to every thread.  red must hold >= 33 doubles.
__device__ __forceinline__ double block_sum(double v, double* red, int tid, int nwarps) {
    int lane = tid & 31, warp = tid >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double s = 0.0;
        if (lane == 0) {
            for (int w = 0; w < nwarps; ++w) s += red[w];
            red[32] = s;
        }
    }
    __syncthreads();
    return red[32];
}

// Block-wide exclusive scan of one u32 per thread; returns the exclusive prefix, *total gets the block sum.
__device__ __forceinline__ u32 block_scan_excl(u32 v, u32* wsum, int tid, int nwarps, u32* total) {
    int lane = tid & 31, warp = tid >> 5;
    u32 inc = warp_scan_incl(v, lane);
    __syncthreads();
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    u32 base = 0, tot = 0;
    for (int w = 0; w < nwarps; ++w) {
        u32 x = wsum[w];
        if (w < warp) base += x;
        tot += x;
    }
    *total = tot;
    return base + inc - v;
}

// =========================================================================================================
// K0: CSR -> bit rows.  One thread per posting (grid-stride); the k-mer of posting p is found by binary
// search in csr_off.  Row 0 stays all-zero (the padding row).
// =========================================================================================================
__global__ void __launch_bounds__(256) build_bitrows_kernel(const u64* __restrict__ csr_off, const u32* __restrict__ csr_ids,
                                                            u64 nnz, const u32* __restrict__ rowmap, u32* __restrict__ bitrows,
                                                            u32 row_words, u64 s0, u64 s1) {
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (u64)gridDim.x * blockDim.x) {
        u32 id = csr_ids[p];
        if (id < s0 || id >= s1) continue;
        u32 lo = 0, hi = 65536;  // largest k with csr_off[k] <= p
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (csr_off[mid] <= p) lo = mid;
            else hi = mid;
        }
        u32 row = rowmap[lo];
        u32 local = (u32)(id - s0);
        atomicOr(&bitrows[(size_t)row * row_words + (local >> 5)], 1u << (local & 31));
    }
}

// =========================================================================================================
// K0 (from sequences): the k-mer -> reference index straight from the lineage-sorted reference sequences, without the
// CSR detour (tree.rs:114-123 windowing, 134-137 unique: setting a bit is idempotent).  Two passes over the 4-bit codes:
//   kmer_presence_kernel     which of the 65 536 8-mers occur in the shard at all (shared-memory bitmap per CTA, OR-ed out)
//   bitrows_from_seq_kernel  bit (row of the k-mer, reference) := 1
// One warp per reference, every lane folds its own windows; a window with an ambiguous base yields nothing (utils.rs:29-38).
// ref_off are offsets into `codes` of the references [ref_first, ref_first + n) of the current upload chunk, rebased to 0.
// =========================================================================================================
__device__ __forceinline__ bool window_kmer(const u8* __restrict__ p, u32* kmer) {
    u32 k = 0;
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const u32 c = p[j];
        ok &= (c == 1u) | (c == 2u) | (c == 4u) | (c == 8u);
        k |= ((u32)(__ffs(c) - 1) & 3u) << (14 - 2 * j);
    }
    *kmer = k;
    return ok;
}

__global__ void __launch_bounds__(256) kmer_presence_kernel(const u64* __restrict__ ref_off, const u8* __restrict__ codes, u32 n, u32* __restrict__ present) {
    __shared__ u32 bitmap[2048];
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < 2048; i += 256) bitmap[i] = 0;
    __syncthreads();
    const u32 warps = gridDim.x * 8u;
    for (u32 r = blockIdx.x * 8u + (tid >> 5); r < n; r += warps) {
        const u64 o = ref_off[r];
        const u32 L = (u32)(ref_off[r + 1] - o);
        for (u32 i = lane; i + 8 <= L; i += 32) {
            u32 k;
            if (window_kmer(codes + o + i, &k)) atomicOr(&bitmap[k >> 5], 1u << (k & 31));
        }
    }
    __syncthreads();
    for (int i = tid; i < 2048; i += 256)
        if (bitmap[i]) atomicOr(&present[i], bitmap[i]);
}

__global__ void __launch_bounds__(256) bitrows_from_seq_kernel(const u64* __restrict__ ref_off, const u8* __restrict__ codes, u32 n, u64 local_first,
                                                               const u32* __restrict__ rowmap, u32* __restrict__ bitrows, u32 row_words) {
    const int tid = threadIdx.x, lane = tid & 31;
    const u32 warps = gridDim.x * 8u;
    for (u32 r = blockIdx.x * 8u + (tid >> 5); r < n; r += warps) {
        const u64 o = ref_off[r];
        const u32 L = (u32)(ref_off[r + 1] - o);
        const u64 local = local_first + r;  // reference id relative to the shard
        const u32 word = (u32)(local >> 5), bit = 1u << (u32)(local & 31);
        for (u32 i = lane; i + 8 <= L; i += 32) {
            u32 k;
            if (window_kmer(codes + o + i, &k)) atomicOr(&bitrows[(size_t)rowmap[k] * row_words + word], bit);
        }
    }
}

// =========================================================================================================
// K1: one CTA (128 threads) per query.  A 65 536-bit bitmap in shared memory is both the dedup set and the
// sort: scanning it in word order emits the unique k-mers ascending (utils.rs:39).
// kmers_both_kernel (--strand both, RTX_BOTH_STRANDS): the same pass also sets rc16(k) in a second bitmap and emits
// the 8-mers of the reverse complement as virtual query n_queries + q.
// =========================================================================================================
constexpr int kKmerThreads = 128;

// the 8-mer of the reverse complement strand at the same window: complement every base (A 0 <-> T 3, C 1 <-> G 2, i.e. x ^ 3)
// and reverse the order of the eight 2-bit groups
__host__ __device__ __forceinline__ u32 rc16(u32 k) {
    u32 x = (k ^ 0xFFFFu) & 0xFFFFu;
    x = ((x >> 2) & 0x3333u) | ((x & 0x3333u) << 2);
    x = ((x >> 4) & 0x0F0Fu) | ((x & 0x0F0Fu) << 4);
    return ((x >> 8) & 0x00FFu) | ((x & 0x00FFu) << 8);
}

// ordered compaction of one 65 536-bit k-mer set into query q's k-mer list, row list, K and padded row count;
// thread t owns bitmap words [16t, 16t+16)
__device__ __forceinline__ void kmers_compact(const IndexView& ix, const BatchView& b, const u32* bitmap, u32* wsum, int q, int tid) {
    u32 cnt = 0, cnt_present = 0;
#pragma unroll
    for (int w = 0; w < 16; ++w) {
        u32 x = bitmap[tid * 16 + w];
        cnt += __popc(x);
        cnt_present += __popc(x & ix.present[tid * 16 + w]);
    }
    u32 total, total_present;
    u32 pos = block_scan_excl(cnt, wsum, tid, kKmerThreads / 32, &total);
    u32 pos2 = block_scan_excl(cnt_present, wsum, tid, kKmerThreads / 32, &total_present);
    u16* kout = b.kmers + (size_t)q * b.kstride;
    u32* rout = b.rows + (size_t)q * b.kstride;
    for (int w = 0; w < 16; ++w) {
        u32 x = bitmap[tid * 16 + w];
        while (x) {
            u32 bit = __ffs(x) - 1;
            x &= x - 1;
            u32 kmer = (u32)(tid * 16 + w) * 32 + bit;
            kout[pos++] = (u16)kmer;
            u32 r = ix.rowmap[kmer];
            if (r) rout[pos2++] = r;
        }
    }
    u32 padded = (total_present + 15u) & ~15u;
    if (tid < 16 && total_present + tid < padded) rout[total_present + tid] = 0;  // zero row
    if (tid == 0) {
        b.K[q] = (u16)total;
        b.nrows[q] = padded;
    }
}

__global__ void __launch_bounds__(kKmerThreads) kmers_kernel(IndexView ix, BatchView b) {
    __shared__ u32 bitmap[2048];
    __shared__ u32 wsum[kKmerThreads / 32];
    const int q = blockIdx.x, tid = threadIdx.x;
    const u64 base = b.seq_off[q];
    const u32 L = (u32)(b.seq_off[q + 1] - base);
    for (int i = tid; i < 2048; i += kKmerThreads) bitmap[i] = 0;
    __syncthreads();
    if (L >= 8) {
        for (u32 i = tid; i + 8 <= L; i += kKmerThreads) {  // sequence.windows(8)
            u32 k = 0;
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                u32 c = b.codes[base + i + j];
                ok &= (c == 1u) | (c == 2u) | (c == 4u) | (c == 8u);  // map_four_to_two_bit_repr -> Some
                k |= ((u32)(__ffs(c) - 1) & 3u) << (14 - 2 * j);      // first base in bits 15..14
            }
            if (ok) atomicOr(&bitmap[k >> 5], 1u << (k & 31));
        }
    }
    __syncthreads();
    // ordered compaction; thread t owns bitmap words [16t, 16t+16)
    u32 cnt = 0, cnt_present = 0;
#pragma unroll
    for (int w = 0; w < 16; ++w) {
        u32 x = bitmap[tid * 16 + w];
        cnt += __popc(x);
        cnt_present += __popc(x & ix.present[tid * 16 + w]);
    }
    u32 total, total_present;
    u32 pos = block_scan_excl(cnt, wsum, tid, kKmerThreads / 32, &total);
    u32 pos2 = block_scan_excl(cnt_present, wsum, tid, kKmerThreads / 32, &total_present);
    u16* kout = b.kmers + (size_t)q * b.kstride;
    u32* rout = b.rows + (size_t)q * b.kstride;
    for (int w = 0; w < 16; ++w) {
        u32 x = bitmap[tid * 16 + w];
        while (x) {
            u32 bit = __ffs(x) - 1;
            x &= x - 1;
            u32 kmer = (u32)(tid * 16 + w) * 32 + bit;
            kout[pos++] = (u16)kmer;
            u32 r = ix.rowmap[kmer];
            if (r) rout[pos2++] = r;
        }
    }
    u32 padded = (total_present + 15u) & ~15u;
    if (tid < 16 && total_present + tid < padded) rout[total_present + tid] = 0;  // zero row
    if (tid == 0) {
        b.K[q] = (u16)total;
        b.nrows[q] = padded;
    }
}

// The window fold is written out again here rather than shared with kmers_kernel through a template or helper: the shared forms
// compile kmers_kernel to different sm_100a code (16 more instructions: the compiler no longer keeps the warp index bound through
// the helper), and the plus-mode kernel is meant to stay exactly as it is.  A change to the fold goes into both kernels.
__global__ void __launch_bounds__(kKmerThreads) kmers_both_kernel(IndexView ix, BatchView b) {
    __shared__ u32 bitmap[2 * 2048];  // [0, 2048) the query's 8-mers, [2048, 4096) those of its reverse complement
    __shared__ u32 wsum[kKmerThreads / 32];
    const int q = blockIdx.x, tid = threadIdx.x;
    const u64 base = b.seq_off[q];
    const u32 L = (u32)(b.seq_off[q + 1] - base);
    for (int i = tid; i < 2 * 2048; i += kKmerThreads) bitmap[i] = 0;
    __syncthreads();
    if (L >= 8) {
        for (u32 i = tid; i + 8 <= L; i += kKmerThreads) {  // sequence.windows(8)
            u32 k = 0;
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                u32 c = b.codes[base + i + j];
                ok &= (c == 1u) | (c == 2u) | (c == 4u) | (c == 8u);
                k |= ((u32)(__ffs(c) - 1) & 3u) << (14 - 2 * j);
            }
            if (ok) {
                atomicOr(&bitmap[k >> 5], 1u << (k & 31));
                const u32 r = rc16(k);
                atomicOr(&bitmap[2048 + (r >> 5)], 1u << (r & 31));
            }
        }
    }
    __syncthreads();
    kmers_compact(ix, b, bitmap, wsum, q, tid);
    kmers_compact(ix, b, bitmap + 2048, wsum, (int)b.n_queries + q, tid);
}

// =========================================================================================================
// K2: hit counting by positional popcount.
//
// count[r] = |kmers(q) ∩ kmers(ref r)| = column sum over the query's bit rows.  Each lane owns kLaneWords consecutive
// 32-bit words of the row (64 references) and keeps the column sums bit-sliced: plane p of a word holds bit p
// of the 32 counters.  16 rows are folded per step with a carry-save adder tree (15 full adders = 30 LOP3)
// whose single weight-16 carry ripples into the high planes.  The epilogue transposes the planes into 32 u16
// counters with a 16x16 bit-matrix transpose done on both half-words at once, stores them and feeds the
// shared-memory histogram.
// =========================================================================================================
constexpr int kHitThreads = 256;
constexpr int kLaneWords = 2;      // words of a row per lane: one 8-byte load per row, a warp tile is 64 words = 2048 references
constexpr int kRowListCap = 4096;  // row ids staged in shared memory per chunk

__device__ __forceinline__ void csa(u32& s, u32& c, u32 a, u32 b, u32 d) {
    u32 x = a ^ b;
    c = (a & b) | (x & d);
    s = x ^ d;
}

// 16 rows into the planes 0..3; the weight-16 carry is returned, not rippled (two of them are merged first, see fold32)
template <int NP>
__device__ __forceinline__ u32 add16_carry(u32 (&pl)[NP], const u32 (&x)[16]) {
    u32 a[8], b4[4], d2[2], e;
#pragma unroll
    for (int i = 0; i < 8; ++i) csa(pl[0], a[i], pl[0], x[2 * i], x[2 * i + 1]);
#pragma unroll
    for (int i = 0; i < 4; ++i) csa(pl[1], b4[i], pl[1], a[2 * i], a[2 * i + 1]);
#pragma unroll
    for (int i = 0; i < 2; ++i) csa(pl[2], d2[i], pl[2], b4[2 * i], b4[2 * i + 1]);
    csa(pl[3], e, pl[3], d2[0], d2[1]);
    return e;
}
// ripple a carry of weight 2^P0 into the planes P0..NP-1
template <int NP, int P0>
__device__ __forceinline__ void ripple(u32 (&pl)[NP], u32 e) {
#pragma unroll
    for (int p = P0; p < NP; ++p) {
        u32 t = pl[p] & e;
        pl[p] ^= e;
        e = t;
    }
}
// two weight-16 carries: one full adder into plane 4, then a single ripple from plane 5
template <int NP>
__device__ __forceinline__ void merge_carries(u32 (&pl)[NP], u32 ea, u32 eb) {
    if (NP > 4) {
        u32 c;
        csa(pl[4 < NP ? 4 : 0], c, pl[4 < NP ? 4 : 0], ea, eb);
        ripple<NP, 5>(pl, c);
    }
}

// planes -> 32 u16 counters packed as 16 words: out[i] = count[2i] | count[2i+1] << 16
template <int NP>
__device__ __forceinline__ void planes_to_counts(const u32 (&pl)[NP], u32 (&out)[16]) {
    u32 A[16];
#pragma unroll
    for (int p = 0; p < 16; ++p) A[p] = (p < NP) ? pl[p] : 0u;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const int j = 8 >> s;
        const u32 m = (s == 0) ? 0x00FF00FFu : (s == 1) ? 0x0F0F0F0Fu : (s == 2) ? 0x33333333u : 0x55555555u;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            if (k & j) continue;
            u32 t = ((A[k] >> j) ^ A[k + j]) & m;
            A[k + j] ^= t;
            A[k] ^= t << j;
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        out[i] = __byte_perm(A[2 * i], A[2 * i + 1], 0x5410);      // references 2i, 2i+1
        out[8 + i] = __byte_perm(A[2 * i], A[2 * i + 1], 0x7632);  // references 16+2i, 16+2i+1
    }
}

__device__ __forceinline__ u32 vec_get(const uint2& v, int i) { return i == 0 ? v.x : v.y; }

// grid: x = query within the sub-batch, y = tile group.  block: 32 * nwarps threads (nwarps chosen by the host so that
// the tiles of a CTA divide evenly over its warps).
// dynamic shared memory: u32 srow[kRowListCap] + u32 shist[hstride]
// The next 16 rows are requested before the current 16 are folded (register double buffer).
// address of a row's slice: one IMAD.WIDE on the fma pipe (the compiler's own choice, IMAD.WIDE + two LEAs, put a third of
// the inner loop's alu-pipe work into address arithmetic; LOP3 shares that pipe at half rate)
__device__ __forceinline__ const void* row_ptr(const u32* __restrict__ colbase, u32 rid, u32 row_bytes) {
    u64 a;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(a) : "r"(rid), "r"(row_bytes), "l"(colbase));
    return reinterpret_cast<const void*>(a);
}
// 16 row ids of the list as four broadcast LDS.128 (one data-pipe wavefront per four rows instead of one per row: with 256 B per row
// and warp the per-row LDS.32 was a third of the L1 data-pipe wavefronts, the unit this kernel saturates first).  j % 16 == 0 and the
// lists start 16-byte aligned (kstride % 16 == 0).
__device__ __forceinline__ void row_ids16(u32 (&r)[16], const u32* __restrict__ srow, u32 j) {
    const uint4* p = reinterpret_cast<const uint4*>(srow + j);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint4 t = p[i];
        r[4 * i] = t.x, r[4 * i + 1] = t.y, r[4 * i + 2] = t.z, r[4 * i + 3] = t.w;
    }
}
__device__ __forceinline__ void load16(uint2 (&x)[16], const u32* __restrict__ colbase, const u32* __restrict__ srow, u32 j, u32 row_bytes) {
    u32 r[16];
    row_ids16(r, srow, j);
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = ldg_stream(reinterpret_cast<const uint2*>(row_ptr(colbase, r[i], row_bytes)));
}

template <int NP>
__device__ __forceinline__ void fold16_carry(u32 (&pl)[kLaneWords][NP], const uint2 (&x)[16], u32 (&e)[kLaneWords]) {
#pragma unroll
    for (int v = 0; v < kLaneWords; ++v) {
        u32 xv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) xv[i] = vec_get(x[i], v);
        e[v] = add16_carry<NP>(pl[v], xv);
    }
}
template <int NP>
__device__ __forceinline__ void merge_carries_v(u32 (&pl)[kLaneWords][NP], const u32 (&ea)[kLaneWords], const u32 (&eb)[kLaneWords]) {
#pragma unroll
    for (int v = 0; v < kLaneWords; ++v) merge_carries<NP>(pl[v], ea[v], eb[v]);
}

// The count vectors (2 * N bytes per query, tens of GB per launch) are written once and read back much later, if at all: streaming
// stores (evict-first) keep them from pushing the L2-blocked slice of the bit matrix out of the L2.
__device__ __forceinline__ void store_counts(uint4* p, const uint4& v) { __stcs(p, v); }

template <int NP>
__global__ void __launch_bounds__(kHitThreads)
    hitcount_bitrows_kernel(IndexView ix, BatchView b, u16* __restrict__ counts, int q_base, int tiles_per_cta, int n_tiles, int hist_global) {
    constexpr int V = kLaneWords;
    extern __shared__ __align__(16) u32 hsm[];
    u32* srow = hsm;
    // hist_global: queries with tens of thousands of 8-mers, whose histogram does not fit shared memory: bins are bumped in global memory
    u32* shist = hist_global ? b.hist + (size_t)(q_base + blockIdx.x) * b.hstride : hsm + kRowListCap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nthreads = blockDim.x, nwarps = nthreads >> 5;
    const int ql = blockIdx.x;
    const int q = q_base + ql;
    const u32 n = b.nrows[q];
    const u32* __restrict__ qrows = b.rows + (size_t)q * b.kstride;
    const int tile_begin = blockIdx.y * tiles_per_cta;
    const int tile_end = min(n_tiles, tile_begin + tiles_per_cta);
    const int rounds = (tile_end - tile_begin + nwarps - 1) / nwarps;
    const u32 nbins = (u32)b.K[q] + 1u;
    const u32 row_bytes = ix.row_words * 4u;

    if (!hist_global)
        for (u32 i = tid; i < nbins; i += nthreads) shist[i] = 0;
    const bool single = n <= (u32)kRowListCap;
    if (single) {
        for (u32 i = tid; i < n; i += nthreads) srow[i] = qrows[i];
    }
    __syncthreads();

    u16* __restrict__ qcounts = counts + (size_t)ql * ix.n_pad;
    for (int r = 0; r < rounds; ++r) {
        const int tile = tile_begin + r * nwarps + warp;
        const bool active = tile < tile_end;
        const u32 word0 = (u32)tile * (32 * V) + lane * V;  // first word of this lane
        u32 pl[V][NP];
#pragma unroll
        for (int v = 0; v < V; ++v)
#pragma unroll
            for (int p = 0; p < NP; ++p) pl[v][p] = 0;

        for (u32 c0 = 0; c0 < n; c0 += kRowListCap) {
            const u32 cn = min((u32)kRowListCap, n - c0);
            if (!single) {
                __syncthreads();
                for (u32 i = tid; i < cn; i += nthreads) srow[i] = qrows[c0 + i];
                __syncthreads();
            }
            if (active) {
                const u32* __restrict__ colbase = ix.bitrows + word0;
                uint2 xa[16], xb[16];
                load16(xa, colbase, srow, 0, row_bytes);
                for (u32 j = 0; j < cn; j += 32) {
                    const bool has_b = j + 16 < cn;
                    u32 ea[V], eb[V];
                    if (has_b) load16(xb, colbase, srow, j + 16, row_bytes);
                    fold16_carry<NP>(pl, xa, ea);
                    if (j + 32 < cn) load16(xa, colbase, srow, j + 32, row_bytes);
                    if (has_b) fold16_carry<NP>(pl, xb, eb);
                    else {
#pragma unroll
                        for (int v = 0; v < V; ++v) eb[v] = 0;
                    }
                    merge_carries_v<NP>(pl, ea, eb);
                }
            }
        }
        if (active) {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                u32 out[16];
                planes_to_counts<NP>(pl[v], out);
                const u64 ref0 = (u64)(word0 + v) * 32;
                uint4* dst = reinterpret_cast<uint4*>(qcounts + ref0);
#pragma unroll
                for (int i = 0; i < 4; ++i) store_counts(dst + i, make_uint4(out[4 * i], out[4 * i + 1], out[4 * i + 2], out[4 * i + 3]));
                if (ref0 + 32 <= ix.shard_refs) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        atomicAdd(&shist[out[i] & 0xFFFFu], 1u);
                        atomicAdd(&shist[out[i] >> 16], 1u);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        if (ref0 + 2 * i < ix.shard_refs) atomicAdd(&shist[out[i] & 0xFFFFu], 1u);
                        if (ref0 + 2 * i + 1 < ix.shard_refs) atomicAdd(&shist[out[i] >> 16], 1u);
                    }
                }
            }
        }
    }
    __syncthreads();
    if (hist_global) return;
    u32* __restrict__ ghist = b.hist + (size_t)q * b.hstride;
    for (u32 i = tid; i < nbins; i += nthreads) {
        u32 h = shist[i];
        if (h) atomicAdd(&ghist[i], h);
    }
}

// =========================================================================================================
// K2 (query-group form): the single-query kernel above sits exactly on the L2 -> SM bandwidth cap (every bit row of every
// query is fetched from L2 once per reference tile: 82 GB per 10 k queries on C2 = 12.4 TB/s).  Queries of one batch share
// rows (two COI queries have ~22 % of their 8-mers in common; the union of 16 queries' rows is ~half the sum), so here a
// CTA carries G queries -- one per warp -- over the SAME reference tile.  The row loads allocate in the L1 (plain
// ld.global.nc), so that a row that another warp of the CTA has fetched shortly before hits there instead of going to the L2.
// The warps run independently, with no block barrier: keeping them in step over the row-id space raises the L1 hit rate but
// the barriers cost more than the hits save (DESIGN.md §4, K2).
// grid: x = query group (fastest: L2 blocking over reference tile groups as before), y = tile group.
// dynamic smem: u32 srow[G][kstride] | u32 shist[G][hstride]
// =========================================================================================================
__device__ __forceinline__ uint2 ldg_l1(const uint2* p) {
    uint2 r;
    asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void load16_l1(uint2 (&x)[16], const u32* __restrict__ colbase, const u32* __restrict__ srow, u32 j) {
    u32 r[16];
    row_ids16(r, srow, j);
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = ldg_l1(reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(colbase) + (u64)r[i] * 512u));
}

constexpr int kHitGroupMaxThreads = 512;

// (A 96-register build, 5 CTAs x 4 warps per SM instead of 4 x 4, spills and measured 6 % slower.)
template <int NP>
__global__ void __launch_bounds__(kHitGroupMaxThreads, 1)
    hitcount_group_kernel(IndexView ix, BatchView b, u16* __restrict__ counts, int q_base, int q_count, int tiles_per_cta, int n_tiles,
                          u16* __restrict__ segmax, size_t segmax_stride) {
    constexpr int V = kLaneWords;
    extern __shared__ __align__(16) u32 hsm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = blockDim.x >> 5;
    u32* srow = hsm + (size_t)warp * b.kstride;
    u32* shist = hsm + (size_t)G * b.kstride + (size_t)warp * b.hstride;
    const int ql = blockIdx.x * G + warp;
    const bool valid = ql < q_count;
    const int q = q_base + (valid ? ql : 0);
    const u32 n = valid ? b.nrows[q] : 0u;  // padded to a multiple of 16 with the all-zero row 0
    const u32 nbins = valid ? (u32)b.K[q] + 1u : 0u;
    const u32* __restrict__ qrows = b.rows + (size_t)q * b.kstride;
    // staged as row offsets in 512-byte units (rows are padded to 128 words), so that the address of a row's slice is ONE
    // IMAD.WIDE.U32 with an immediate multiplier (with the row size in a uniform register ptxas emits IMAD.WIDE + IADD3 + IMAD.X)
    const u32 row_units = ix.row_words >> 7;
    for (u32 i = lane; i < n; i += 32) srow[i] = qrows[i] * row_units;
    for (u32 i = lane; i < nbins; i += 32) shist[i] = 0;
    __syncwarp();

    const int tile_begin = blockIdx.y * tiles_per_cta;
    const int tile_end = min(n_tiles, tile_begin + tiles_per_cta);
    u16* __restrict__ qcounts = counts + (size_t)ql * ix.n_pad;
    for (int tile = tile_begin; tile < tile_end; ++tile) {
        const u32 word0 = (u32)tile * (32 * V) + lane * V;
        const u32* __restrict__ colbase = ix.bitrows + word0;
        u32 pl[V][NP];
#pragma unroll
        for (int v = 0; v < V; ++v)
#pragma unroll
            for (int p = 0; p < NP; ++p) pl[v][p] = 0;
        uint2 xa[16], xb[16];
        if (n) load16_l1(xa, colbase, srow, 0);
        for (u32 j = 0; j < n; j += 32) {
            const bool has_b = j + 16 < n;
            u32 ea[V], eb[V];
            if (has_b) load16_l1(xb, colbase, srow, j + 16);
            fold16_carry<NP>(pl, xa, ea);
            if (j + 32 < n) load16_l1(xa, colbase, srow, j + 32);
            if (has_b) fold16_carry<NP>(pl, xb, eb);
            else {
#pragma unroll
                for (int v = 0; v < V; ++v) eb[v] = 0;
            }
            merge_carries_v<NP>(pl, ea, eb);
        }
        if (valid) {
            u32 lane_max = 0;  // largest count among this lane's 32 * V references, in both half-words
#pragma unroll
            for (int v = 0; v < V; ++v) {
                u32 out[16];
                planes_to_counts<NP>(pl[v], out);
                u32 word_max = 0;
#pragma unroll
                for (int i = 0; i < 16; ++i) word_max = __vmaxu2(word_max, out[i]);
                lane_max = __vmaxu2(lane_max, word_max);
                const u64 ref0 = (u64)(word0 + v) * 32;
                uint4* dst = reinterpret_cast<uint4*>(qcounts + ref0);
#pragma unroll
                for (int i = 0; i < 4; ++i) store_counts(dst + i, make_uint4(out[4 * i], out[4 * i + 1], out[4 * i + 2], out[4 * i + 3]));
                if (ref0 + 32 <= ix.shard_refs) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        atomicAdd(&shist[out[i] & 0xFFFFu], 1u);
                        atomicAdd(&shist[out[i] >> 16], 1u);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        if (ref0 + 2 * i < ix.shard_refs) atomicAdd(&shist[out[i] & 0xFFFFu], 1u);
                        if (ref0 + 2 * i + 1 < ix.shard_refs) atomicAdd(&shist[out[i] >> 16], 1u);
                    }
                }
            }
            // largest count per 512-reference prefix segment (32 * V = 64 references per lane: 8 lanes per segment), so that K4 can
            // drop a segment below m_min without reading its counts (padding references count 0 and never raise the maximum)
            if (segmax != nullptr) {
                u32 m = max(lane_max & 0xFFFFu, lane_max >> 16);
                constexpr int kLanesPerSeg = 512 / (32 * V);
#pragma unroll
                for (int o = 1; o < kLanesPerSeg; o <<= 1) m = max(m, __shfl_xor_sync(kFullMask, m, o));
                if ((lane & (kLanesPerSeg - 1)) == 0)
                    segmax[(size_t)ql * segmax_stride + (size_t)tile * (32 / kLanesPerSeg) + lane / kLanesPerSeg] = (u16)m;
            }
        }
    }
    __syncwarp();
    if (valid) {
        u32* __restrict__ ghist = b.hist + (size_t)q * b.hstride;
        for (u32 i = lane; i < nbins; i += 32) {
            const u32 h = shist[i];
            if (h) atomicAdd(&ghist[i], h);
        }
    }
}

// =========================================================================================================
// K2 (variant): the reference's own data structure -- CSR postings with u32 ids (tree.rs:22,41) walked per
// query k-mer, counters in shared memory.  One CTA per (query, reference tile of kCsrTileRefs references);
// u16 counters are packed two per 32-bit word so that neighbouring ids hit neighbouring banks.
// =========================================================================================================
constexpr int kCsrThreads = 256;
constexpr int kCsrTileRefs = 65536;  // 128 KB of packed u16 counters

__global__ void __launch_bounds__(kCsrThreads)
    hitcount_csr_kernel(IndexView ix, BatchView b, u16* __restrict__ counts, int q_base) {
    extern __shared__ __align__(16) u32 csm[];
    u32* cnt = csm;                          // [kCsrTileRefs / 2]
    u32* shist = csm + kCsrTileRefs / 2;     // [hstride]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ql = blockIdx.x, q = q_base + ql;
    const u64 tile0 = ix.shard_begin + (u64)blockIdx.y * kCsrTileRefs;  // global id range of this tile
    const u64 tile1 = min(ix.shard_begin + ix.shard_refs, tile0 + kCsrTileRefs);
    const u32 K = b.K[q];
    const u32 nbins = K + 1u;
    for (u32 i = tid; i < kCsrTileRefs / 2; i += kCsrThreads) cnt[i] = 0;
    for (u32 i = tid; i < nbins; i += kCsrThreads) shist[i] = 0;
    __syncthreads();
    const u16* __restrict__ kmers = b.kmers + (size_t)q * b.kstride;
    // one warp per posting list; the sub-range falling into the tile is found by binary search (lists ascend)
    for (u32 ki = warp; ki < K; ki += kCsrThreads / 32) {
        const u32 kmer = kmers[ki];
        u64 o0 = ix.csr_off[kmer], o1 = ix.csr_off[kmer + 1];
        u64 lo = o0, hi = o1;  // first posting >= tile0
        while (lo < hi) {
            u64 mid = (lo + hi) >> 1;
            if (ix.csr_ids[mid] < tile0) lo = mid + 1;
            else hi = mid;
        }
        const u64 a = lo;
        hi = o1;  // first posting >= tile1
        while (lo < hi) {
            u64 mid = (lo + hi) >> 1;
            if (ix.csr_ids[mid] < tile1) lo = mid + 1;
            else hi = mid;
        }
        const u64 e = lo;
        for (u64 p = a + lane; p < e; p += 32) {
            u32 local = (u32)(ix.csr_ids[p] - tile0);
            atomicAdd(&cnt[local >> 1], (local & 1u) ? 0x10000u : 1u);
        }
    }
    __syncthreads();
    u16* __restrict__ qcounts = counts + (size_t)ql * ix.n_pad + (tile0 - ix.shard_begin);
    const u32 nref = (u32)(tile1 - tile0);
    u32* qc32 = reinterpret_cast<u32*>(qcounts);
    for (u32 i = tid; i < (nref + 1) / 2; i += kCsrThreads) {
        u32 w = cnt[i];
        qc32[i] = w;
        atomicAdd(&shist[w & 0xFFFFu], 1u);
        if (2 * i + 1 < nref) atomicAdd(&shist[w >> 16], 1u);
    }
    __syncthreads();
    u32* __restrict__ ghist = b.hist + (size_t)q * b.hstride;
    for (u32 i = tid; i < nbins; i += kCsrThreads) {
        u32 h = shist[i];
        if (h) atomicAdd(&ghist[i], h);
    }
}

// =========================================================================================================
// K2': --skip-exact-matches (raxtax.rs:65-68): counter of every exact match := 0, histogram adjusted.
// One thread per query of the sub-batch.
// =========================================================================================================
__global__ void fixup_exact_kernel(IndexView ix, BatchView b, u16* __restrict__ counts, int q_base, int q_count) {
    int ql = blockIdx.x * blockDim.x + threadIdx.x;
    if (ql >= q_count || b.exact_off == nullptr) return;
    int q = q_base + ql;
    u32* hist = b.hist + (size_t)q * b.hstride;
    for (u32 e = b.exact_off[q]; e < b.exact_off[q + 1]; ++e) {
        u64 id = b.exact_ids[e];
        if (id < ix.shard_begin || id >= ix.shard_begin + ix.shard_refs) continue;
        u16* c = counts + (size_t)ql * ix.n_pad + (id - ix.shard_begin);
        u16 old = *c;
        if (old != 0) {
            *c = 0;
            atomicSub(&hist[old], 1u);
            atomicAdd(&hist[0], 1u);
        }
    }
}

// =========================================================================================================
// K2'' (--strand both, RTX_BOTH_STRANDS): the orientation of every query of the sub-batch.  M(x), the largest hit count of
// strand x after the skip zeroing, is the top non-empty bucket of x's histogram; the query is classified as its reverse
// complement (virtual query n + q) iff M(rc) > M(fwd), every tie stays forward.  For a reverse winner this kernel leaves in
// query q's place what K3-K5 and the taps read: the histogram row, the k-mer list, the count row and the per-segment maxima
// (K is the same for both strands).  One CTA per query.
// =========================================================================================================
constexpr int kStrandThreads = 256;

__global__ void __launch_bounds__(kStrandThreads, 1)
    strand_select_kernel(IndexView ix, BatchView b, u16* __restrict__ counts, const u16* __restrict__ counts_rc, u16* __restrict__ segmax,
                         size_t segmax_stride, const u16* __restrict__ segmax_rc, u32 n_seg, u8* __restrict__ strand, int q_base) {
    __shared__ u32 smax[2];
    const int tid = threadIdx.x, ql = blockIdx.x;
    const int q = q_base + ql, qr = (int)b.n_queries + q;
    const u32 K = b.K[q];
    u32* __restrict__ hf = b.hist + (size_t)q * b.hstride;
    const u32* __restrict__ hr = b.hist + (size_t)qr * b.hstride;
    if (tid < 2) smax[tid] = 0;
    __syncthreads();
    u32 mf = 0, mr = 0;
    for (u32 i = tid; i <= K; i += kStrandThreads) {  // ascending per thread: the last non-empty bucket seen is the thread's largest
        if (hf[i]) mf = i;
        if (hr[i]) mr = i;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mf = max(mf, __shfl_xor_sync(kFullMask, mf, o));
        mr = max(mr, __shfl_xor_sync(kFullMask, mr, o));
    }
    if ((tid & 31) == 0) {
        atomicMax(&smax[0], mf);
        atomicMax(&smax[1], mr);
    }
    __syncthreads();
    const bool rc = smax[1] > smax[0];
    if (tid == 0) strand[q] = rc ? 1 : 0;
    if (!rc) return;
    for (u32 i = tid; i <= K; i += kStrandThreads) hf[i] = hr[i];
    u16* __restrict__ kf = b.kmers + (size_t)q * b.kstride;
    const u16* __restrict__ kr = b.kmers + (size_t)qr * b.kstride;
    for (u32 i = tid; i < K; i += kStrandThreads) kf[i] = kr[i];
    // count rows: n_pad is a multiple of 4096 references, so whole 16-byte vectors
    uint4* __restrict__ cf = reinterpret_cast<uint4*>(counts + (size_t)ql * ix.n_pad);
    const uint4* __restrict__ cr = reinterpret_cast<const uint4*>(counts_rc + (size_t)ql * ix.n_pad);
    for (u64 i = tid; i < ix.n_pad / 8; i += kStrandThreads) cf[i] = cr[i];
    if (segmax_rc != nullptr)
        for (u32 s = tid; s < n_seg; s += kStrandThreads) segmax[(size_t)ql * segmax_stride + s] = segmax_rc[(size_t)ql * n_seg + s];
}

// The exact matches of the classified orientation, as the override of the tree walk reads them (raxtax.rs:42,73-84):
// sel_off[q + 1] = sel_off[q] + |exact matches of q's classified strand| over the sub-batch [q_base, q_base + q_count), ids behind.
// The batch's exact_off / exact_ids hold the forward strands at [0, n) and the reverse complements at [n, 2n).  One CTA; the
// sub-batches run in order on one stream, so sel_off[q_base] is already written (0 for the first).
constexpr int kStrandScanThreads = 1024;

__global__ void __launch_bounds__(kStrandScanThreads)
    strand_exact_kernel(BatchView b, const u8* __restrict__ strand, u32* __restrict__ sel_off, u32* __restrict__ sel_ids, int q_base, int q_count) {
    __shared__ u32 wsum[kStrandScanThreads / 32];
    __shared__ u32 carry;
    const int tid = threadIdx.x;
    if (tid == 0) {
        if (q_base == 0) sel_off[0] = 0;
        carry = q_base == 0 ? 0u : sel_off[q_base];
    }
    __syncthreads();
    for (int c0 = 0; c0 < q_count; c0 += kStrandScanThreads) {
        const int ql = c0 + tid;
        u32 src = 0, len = 0;
        if (ql < q_count) {
            const int q = q_base + ql;
            const u32 s = strand[q] ? b.n_queries + (u32)q : (u32)q;
            src = b.exact_off[s];
            len = b.exact_off[s + 1] - src;
        }
        u32 total;
        const u32 pos = carry + block_scan_excl(len, wsum, tid, kStrandScanThreads / 32, &total);
        if (ql < q_count) {
            sel_off[q_base + ql + 1] = pos + len;
            for (u32 e = 0; e < len; ++e) sel_ids[pos + e] = b.exact_ids[src + e];
        }
        __syncthreads();
        if (tid == 0) carry += total;
        __syncthreads();
    }
}

// =========================================================================================================
// K3: highest-hit probabilities (prob.rs:8-103).  Persistent CTAs (256 threads), one query at a time.
//
// The reference evaluates, for every distinct count m, the log-pmf p_m(i), its log-cmf c_m(i) and
//   P(m) = sum_i exp(p_m(i) + prod(i) - c_m(i)),   prod(i) = sum_m' h[m'] c_m'(i)            (prob.rs:43-91)
// over the full D x (t+1) grid.  Almost all of that grid cannot influence a result digit:
//   * E(i) = exp(prod(i)) is a product of cmfs, non-decreasing in i, and sum_r P_r >= 1 (some reference always attains
//     the maximum), so every term with E(i) < e^-70 changes a normalised probability by < 1e-30.  An upper bound
//     B(i) >= prod(i) with a closed form per row (geometric bound of the cmf below the mode, -pmf(i+1) above it) is
//     searched for the largest i with B(i) <= -70; everything below i0 = i + 1 is skipped (E := 0).
//   * above its mode the pmf is log-concave and decays geometrically; once p_m(i) < -(40 + ln h[m]) the remaining tail
//     changes neither c_m (h[m]*tail < 1e-17) nor P(m) (tail < 1e-17/h[m]).  That index hi_m is found by a warp-wide
//     search on the closed form.
// What is left per row is the window [i0, hi_m): empty for the bulk of the references (their tail is gone long
// before E wakes up), a few dozen entries for the rows in between (evaluated from the top: cmf = 1 - sf, c = log1p(-sf)),
// and a forward cmf from the first representable pmf for the few rows whose mode lies above i0.
// Result: the same normalised probabilities to ~1e-13 absolute (tests pin 1e-6) at a fraction of the ln/exp count.
// =========================================================================================================
constexpr int kProbThreads = 256;
constexpr int kProbWarps = kProbThreads / 32;
constexpr double kEcut = 70.0;       // E(i) < e^-70 is dropped
constexpr float kTailNats = 40.0f;   // pmf tail cut-off: p < -(kTailNats + ln h)

struct ProbScratch {
    double* cbuf;        // [slots][cbuf_stride] r_m[i] = pmf_m(i) / cmf_m(i) of the slow branch, row d = distinct count d
    size_t cbuf_stride;  // = hstride * tstride doubles
    u32 tstride;         // doubles per cbuf row ( >= max t + 1 )
    double* blk;         // [sub-batch queries][blk_stride] prefix sum of the normalised probabilities at the start of every block of 8
    size_t blk_stride;   //   references, relative to the start of the block's 512-reference segment (K4 -> walk)
    const u16* counts;   // [sub-batch queries][counts_stride] the slot's count vectors (K2 -> K4, walk)
    size_t counts_stride;
    u32 hstride;         // stride of ptab
    double* segoff;      // [sub-batch queries][segoff_stride] prefix sum at the start of every 512-reference segment
    size_t segoff_stride;
    u32 seg_aux_off;     // per query, behind the segment offsets (in doubles): u32 aux[] = { m_min, 0, skip bitmap words ..., u16 segmax[n_seg] }
                         //   segmax (K2 -> K4): largest count of every 512-reference segment
                         //   m_min (K3 -> K4): counts below it carry < kMassCut of the probability mass altogether and are taken as 0
                         //   skip bit s (K4 -> walk): no reference of segment s reaches m_min; its block prefixes were not written
    double* ptab;        // [sub-batch queries][hstride] normalised P(m), direct-indexed by count (K3 -> K4)
    int nprod;           // kProbWarps: one partial prod array per warp; 1: a single array updated with shared-memory atomics
    int lf_smem;         // 1: ln n! staged in shared memory, 0: read from HBM/L2 (very long queries)
    // queries beyond ~6.4 kb (up to the 65 535 8-mers raxtax.rs:56 allows): the per-query tables of K3 live in global scratch
    // (one slot per CTA, same carve-up as the shared-memory layout) and K4 gathers P(m) from the global table
    unsigned char* big;  // null: tables in shared memory
    size_t big_stride;   // bytes per CTA slot
};

// dynamic smem carve-up (sizes depend on H = hstride, T1 = H/2 + 1)
struct ProbSmem {
    double* lf;     // [H + T1]  ln n! for n < K + t (query independent, loaded once per CTA)
    double* Pd;     // [H]       P(m) per distinct count
    double* prodw;  // [kProbWarps][T1]  per-warp partial sums of h[m] * ln cmf_m(i)
    double* E;      // [T1]      exp(prod(i))
    u32* hist;      // [H]
    u32* dh;        // [H]   multiplicity of distinct count d
    u16* dm;        // [H]   distinct counts ascending
    u16* wlo;       // [H]   per distinct count: window [wlo, whi) of entries stored in cbuf
    u16* whi;       // [H]
    u16* mode;      // [H]   mode of pmf_m per distinct count (the 64-bit division is done once per row)
    __host__ __device__ ProbSmem(unsigned char* base, u32 H, u32 T1, int nprod, int lf_smem) {
        lf = reinterpret_cast<double*>(base);
        Pd = lf + (lf_smem ? H + T1 : 0);
        prodw = Pd + H;
        E = prodw + (size_t)nprod * T1;
        hist = reinterpret_cast<u32*>(E + T1);
        dh = hist + H;
        dm = reinterpret_cast<u16*>(dh + H);
        wlo = dm + H;
        whi = wlo + H;
        mode = whi + H;
    }
    static size_t bytes(u32 H, u32 T1, int nprod, int lf_smem) {
        return (size_t)H * (8 + 4 * 2 + 2 * 4) + (size_t)T1 * 8 * (1 + nprod) + (lf_smem ? (size_t)(H + T1) * 8 : 0) + 64;
    }
};

// node record: one 16-byte load gives everything the walk needs about a child
struct __align__(16) NodeRec {
    u32 blo, bhi;      // [lo, hi) clamped to the shard, as local reference positions
    u32 child_first;
    u32 cc_type;       // child_count | node_type << 30
    u32 slo, shi;      // prefix segments of the references in front of blo / bhi
    u32 lo, size;      // node_lo and node_hi - node_lo (global reference ids, not clamped to the shard)
};

// One query's view of what K4 left behind.  The prefix sums of lineage.rs:61-77 are not materialised per reference (8 * N bytes per
// query) nor per node boundary (5.6 MB per query on 1 M references, which made K4 HBM-write-bound on flat profiles): K4 stores one
// value per 32 references, and whoever needs the mass in front of a position adds the up to 32 values P(count[r]) in between.
struct MassView {
    const double* __restrict__ blk;
    const double* __restrict__ segoff;
    const u32* __restrict__ skipw;
    const u16* __restrict__ counts;
    const double* __restrict__ ptab;
};
__device__ __forceinline__ const u32* seg_aux(const ProbScratch& sc, int ql);
__device__ __forceinline__ MassView mass_view(const ProbScratch& sc, int ql) {
    return MassView{sc.blk + (size_t)ql * sc.blk_stride, sc.segoff + (size_t)ql * sc.segoff_stride, seg_aux(sc, ql) + 2,
                    sc.counts + (size_t)ql * sc.counts_stride, sc.ptab + (size_t)ql * sc.hstride};
}
__device__ __forceinline__ bool seg_skipped(const MassView& m, u32 s) { return (m.skipw[s >> 5] >> (s & 31)) & 1u; }
constexpr u32 kBlkRefs = 8;  // references per stored prefix value
// mass of the local references in front of position p, relative to the start of segment s = segment of reference p - 1 (0 for p == 0)
__device__ __forceinline__ double mass_rel(const MassView& m, u32 p, u32 s) {
    // (the loads are issued before the skip bit is known: one dependent round trip less on the walk's critical path)
    const u32 last = p ? p - 1u : 0u, k = last & 7u;
    const uint4 c = *reinterpret_cast<const uint4*>(m.counts + (last & ~7u));  // the eight counts of the block, one 16-byte load
    double v = m.blk[last >> 3];
    if (p == 0u || seg_skipped(m, s)) return 0.0;  // a skipped segment holds no mass (and stale block prefixes)
    v += m.ptab[c.x & 0xFFFFu];
    if (k >= 1) v += m.ptab[c.x >> 16];
    if (k >= 2) v += m.ptab[c.y & 0xFFFFu];
    if (k >= 3) v += m.ptab[c.y >> 16];
    if (k >= 4) v += m.ptab[c.z & 0xFFFFu];
    if (k >= 5) v += m.ptab[c.z >> 16];
    if (k >= 6) v += m.ptab[c.w & 0xFFFFu];
    if (k >= 7) v += m.ptab[c.w >> 16];
    return v;
}
// confidence of a node = sum of the normalised probabilities of its references (lineage.rs:114-117).  r.blo / r.bhi: the node's
// local reference range (clamped to the shard), r.slo / r.shi: the segments of the references in front of them.
__device__ __forceinline__ double node_conf(const MassView& m, const NodeRec& r) {
    const u32 n = r.bhi - r.blo;
    if (n <= 4u) {  // a few references (at most two segments): their probabilities themselves, in order
        if (n == 0u) return 0.0;
        const u32 sa = r.blo >> 9, sb = (r.bhi - 1u) >> 9;  // kPrefixSeg == 512
        const bool ka = !seg_skipped(m, sa), kb = !seg_skipped(m, sb);
        u32 c[4];
#pragma unroll
        for (u32 i = 0; i < 4; ++i) c[i] = i < n ? (u32)m.counts[r.blo + i] : 0u;
        double v = 0.0;
#pragma unroll
        for (u32 i = 0; i < 4; ++i)
            if (i < n && (((r.blo + i) >> 9) == sa ? ka : kb)) v += m.ptab[c[i]];
        return v;
    }
    return (m.segoff[r.shi] - m.segoff[r.slo]) + (mass_rel(m, r.bhi, r.shi) - mass_rel(m, r.blo, r.slo));
}
__device__ __forceinline__ const u32* seg_aux(const ProbScratch& sc, int ql) {
    return reinterpret_cast<const u32*>(sc.segoff + (size_t)ql * sc.segoff_stride + sc.seg_aux_off);
}
// u16 segmax[n_seg] behind the skip bitmap words (K2 -> K4)
__host__ __device__ __forceinline__ const u16* seg_max(const ProbScratch& sc, int ql, u32 n_seg) {
    return reinterpret_cast<const u16*>(reinterpret_cast<const u32*>(sc.segoff + (size_t)ql * sc.segoff_stride + sc.seg_aux_off) + 2 + (n_seg + 31) / 32);
}
constexpr double kMassCut = 1e-25;

// ln pmf_m(i) = ln C(m+i-1,i) + ln C(K-m+t-i-1,t-i) - ln C(K+t-1,t): closed form of the iterative sums of prob.rs:136-166.
// cm = ln (m-1)! + ln (K-m-1)! + T collects the terms that do not depend on i.   Requires 1 <= m <= K-1, i <= t.
__device__ __forceinline__ double ln_pmf(const double* __restrict__ lf, u32 K, u32 t, u32 m, u32 i, double cm) {
    return (lf[m + i - 1] - lf[i]) + (lf[K - m + t - i - 1] - lf[t - i]) - cm;
}

// mode of pmf_m: the first i with pmf(i+1)/pmf(i) = (m+i)(t-i) / ((i+1)(K-m+t-i-1)) < 1, i.e. i > (m t - K + m - t + 1)/(K - 2)
__device__ __forceinline__ u32 pmf_mode(u32 K, u32 t, u32 m) {
    if (K <= 2) return t;
    const long long num = (long long)m * t - (long long)K + m - (long long)t + 1;
    if (num < 0) return 0;
    const long long q = num / (long long)(K - 2) + 1;
    return (u32)min((long long)t, q);
}

// smallest i in [a, bnd) with pred(i), else bnd; pred is monotone (false.. true..).  Warp-wide 32-ary search.
template <typename Pred>
__device__ __forceinline__ u32 warp_first_true(u32 a, u32 bnd, int lane, Pred pred) {
    while (a < bnd) {
        const u32 s = (bnd - a + 31u) / 32u;
        const u32 x = a + (u32)lane * s;
        const bool tested = x < bnd;
        const bool pr = tested && pred(x);
        const u32 hit = __ballot_sync(kFullMask, pr);
        if (!hit) {
            const u32 tmask = __ballot_sync(kFullMask, tested);
            a = a + (u32)(31 - __clz(tmask)) * s + 1u;  // everything up to the last tested point is false
            continue;
        }
        const u32 j = (u32)__ffs(hit) - 1u;
        if (j == 0) return a;
        bnd = a + j * s;          // pred(bnd) holds
        a = bnd - s + 1u;         // pred(a - 1) does not
    }
    return bnd;
}

template <bool BIG>  // BIG: per-query tables in a global scratch slot (long queries); else shared memory, with shared-memory addressing
__global__ void __launch_bounds__(kProbThreads, 4)
    prob_table_kernel(IndexView ix, BatchView b, ResultPool pool, ProbScratch sc, int q_base, int q_count,
                      unsigned long long* __restrict__ hits_total, unsigned long long* __restrict__ next_query) {
    extern __shared__ __align__(16) unsigned char psm_raw[];
    __shared__ double red[40];
    __shared__ u32 wsum[kProbWarps];
    __shared__ int sflag[kProbWarps];

    const u32 H = b.hstride;
    const u32 T1 = H / 2 + 1;
    ProbSmem sm(BIG ? sc.big + (size_t)blockIdx.x * sc.big_stride : psm_raw, H, T1, sc.nprod, sc.lf_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double NEG_INF = -CUDART_INF;
    const double Nd = (double)ix.n_refs;
    const double* __restrict__ lf = sc.lf_smem ? sm.lf : ix.lnfact;

    double* cbuf = sc.cbuf + (size_t)blockIdx.x * sc.cbuf_stride;
    if (sc.lf_smem)
        for (u32 i = tid; i < H + T1; i += kProbThreads) sm.lf[i] = ix.lnfact[i];
    const bool own_prod = sc.nprod == kProbWarps;
    double* __restrict__ myprod = sm.prodw + (own_prod ? (size_t)warp * T1 : 0);
    auto prod_add = [&](u32 i, double v) {
        if (own_prod) myprod[i] += v;
        else atomicAdd(&myprod[i], v);
    };

    // queries are handed out through a counter: a fast-branch query costs a few microseconds, a slow-branch one up to ~100, and
    // a static round-robin left the CTAs 12 % idle at the tail
    __shared__ int s_next;
    while (true) {
        __syncthreads();  // smem reuse across queries (also orders the previous read of s_next)
        if (tid == 0) s_next = (int)atomicAdd(next_query, 1ull);
        __syncthreads();
        const int ql = s_next;
        if (ql >= q_count) break;
        const int q = q_base + ql;
        const u32 K = b.K[q];
        const u32 t = K / 2;  // raxtax.rs:57
        const u32* __restrict__ ghist = b.hist + (size_t)q * H;
        double* __restrict__ ptab = sc.ptab + (size_t)ql * H;

        // ---- histogram -> distinct counts (ascending), prob.rs:13-19 ------------------------------------
        const u32 per = (K + 1 + kProbThreads - 1) / kProbThreads;
        const u32 m_lo = min(K + 1, (u32)tid * per), m_hi = min(K + 1, m_lo + per);
        u32 nz = 0;
        for (u32 m = m_lo; m < m_hi; ++m) {
            u32 h = ghist[m];
            sm.hist[m] = h;
            nz += (h != 0);
            ptab[m] = 0.0;
        }
        u32 D;
        u32 dpos = block_scan_excl(nz, wsum, tid, kProbWarps, &D);
        for (u32 m = m_lo; m < m_hi; ++m) {
            u32 h = sm.hist[m];
            if (h) {
                sm.dm[dpos] = (u16)m;
                sm.dh[dpos] = h;
                sm.Pd[dpos] = 0.0;
                sm.wlo[dpos] = 0;
                sm.whi[dpos] = 0;
                sm.mode[dpos] = (u16)pmf_mode(K, K / 2, m);
                ++dpos;
            }
        }
        __syncthreads();
        // postings a CSR walk would have touched for this query = sum_r count[r]
        {
            unsigned long long hsum = 0;
            for (u32 d = tid; d < D; d += kProbThreads) hsum += (unsigned long long)sm.dm[d] * sm.dh[d];
            for (int o = 16; o > 0; o >>= 1) hsum += __shfl_xor_sync(kFullMask, hsum, o);
            if (lane == 0 && hsum) atomicAdd(hits_total, hsum);
        }

        // ---- P(m) per distinct count -------------------------------------------------------------------
        const bool any_full = sm.hist[K] > 0;  // prob.rs:24-26 (K == 0: every count equals K)
        // T = ln C(K+t-1, t); for K == 0 the reference's u64 arithmetic wraps and yields 0.0, never used then
        const double T = (K == 0) ? 0.0 : lf[K + t - 1] - lf[t] - lf[K - 1];
        if (any_full) {  // fast branch, only_last_pmf (prob.rs:105-119)
            for (u32 d = tid; d < D; d += kProbThreads) {
                u32 m = sm.dm[d];
                double P;
                if (m == K) P = 1.0;
                else if (m == 0) P = 0.0;
                else P = exp(lf[m + t - 1] - lf[t] - lf[m - 1] - T);
                sm.Pd[d] = P;
            }
        } else {  // slow branch (prob.rs:43-91); here 0 <= m < K for every distinct count
            // ---- i0: everything below has E(i) < e^-kEcut -------------------------------------------------
            int slo = -1, shi = (int)t + 1;  // B(slo) <= -kEcut (or slo == -1); nothing known at or above shi
            while (shi - slo > 1) {
                const int s = max(1, (shi - slo - 1 + kProbWarps - 1) / kProbWarps);
                const int cand = slo + (warp + 1) * s;
                bool ok = false;
                if (cand < shi) {
                    const u32 i = (u32)cand;
                    double bsum = 0.0;
                    for (u32 d = lane; d < D; d += 32) {
                        const u32 m = sm.dm[d];
                        if (m == 0) continue;  // cmf == 1
                        const double cm = lf[m - 1] + lf[K - m - 1] + T;
                        double u;
                        if (i < (u32)sm.mode[d]) {  // cmf(i) <= pmf(i) / (1 - pmf(i-1)/pmf(i)): ratios shrink downwards
                            u = ln_pmf(lf, K, t, m, i, cm);
                            if (i > 0) {
                                const double rd = ((double)i * (double)(K - m + t - i)) / ((double)(m + i - 1) * (double)(t - i + 1));
                                u = (rd < 1.0) ? u - log1p(-rd) : 0.0;
                            }
                            u = fmin(u, 0.0);
                        } else {  // ln cmf = ln(1 - sf) <= -sf <= -pmf(i+1)
                            u = (i + 1 <= t) ? -exp(ln_pmf(lf, K, t, m, i + 1, cm)) : 0.0;
                        }
                        bsum = fma((double)sm.dh[d], u, bsum);
                    }
                    bsum = warp_sum(bsum);
                    ok = bsum <= -kEcut;
                }
                if (lane == 0) sflag[warp] = ok;
                __syncthreads();
                int best = -1;
#pragma unroll
                for (int k = 0; k < kProbWarps; ++k)
                    if (sflag[k]) best = k;
                if (best < 0) shi = min(shi, slo + s);
                else {
                    if (best + 1 < kProbWarps) shi = min(shi, slo + (best + 2) * s);
                    slo = slo + (best + 1) * s;
                }
                __syncthreads();
            }
            const u32 i0 = (u32)(slo + 1);
            for (u32 i = tid; i < (u32)sc.nprod * T1; i += kProbThreads) sm.prodw[i] = 0.0;
            __syncthreads();

            // ---- pass 1: one warp per row, rows dealt in descending m ---------------------------------------
            for (int d = (int)D - 1 - warp; d >= 0; d -= kProbWarps) {
                const u32 m = sm.dm[d];
                if (m == 0) continue;  // pmf = [1,0,..]: cmf == 1, ln cmf == 0, P(0) = E(0)
                const double hd = (double)sm.dh[d];
                const double cm = lf[m - 1] + lf[K - m - 1] + T;
                const u32 mode = sm.mode[d];
                const double thr = -(double)(kTailNats + __logf((float)sm.dh[d]));
                // hi: first i above the mode whose pmf (and, by log-concavity, whole remaining tail) is negligible
                const u32 hi = warp_first_true(mode + 1, t + 1, lane, [&](u32 i) { return ln_pmf(lf, K, t, m, i, cm) < thr; });
                double* __restrict__ row = cbuf + (size_t)d * sc.tstride;
                if (i0 > mode) {  // cmf(i0) >~ 1/2: evaluate from the top, cmf = 1 - sf
                    if (hi <= i0) continue;  // the row is finished before E wakes up: c == 0, P == 0
                    double carry = 0.0;
                    for (int c = (int)((hi - 1) >> 5); c >= (int)(i0 >> 5); --c) {
                        const u32 i = (u32)c * 32 + lane;
                        const bool valid = i >= i0 && i < hi;
                        const double e = valid ? exp(ln_pmf(lf, K, t, m, i, cm)) : 0.0;
                        double sfx = e;  // inclusive suffix sum over the lanes
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const double y = __shfl_down_sync(kFullMask, sfx, o);
                            if (lane + o < 32) sfx += y;
                        }
                        const double sf = (sfx - e) + carry;  // sum_{j > i} pmf(j)
                        carry += __shfl_sync(kFullMask, sfx, 0);
                        if (valid) {
                            prod_add(i, hd * log1p(-sf));
                            row[i] = e / (1.0 - sf);
                        }
                    }
                    if (lane == 0) {
                        sm.wlo[d] = (u16)i0;
                        sm.whi[d] = (u16)hi;
                    }
                } else {  // forward from the first representable pmf, as the reference's running sum
                    const u32 lo = warp_first_true(0u, mode + 1, lane, [&](u32 i) { return ln_pmf(lf, K, t, m, i, cm) > -745.0; });
                    double S = 0.0;
                    for (u32 c = lo >> 5; c <= ((hi - 1) >> 5); ++c) {
                        const u32 i = c * 32 + lane;
                        const bool valid = i >= lo && i < hi;
                        const double e = valid ? exp(ln_pmf(lf, K, t, m, i, cm)) : 0.0;
                        const double inc = warp_scan_incl(e, lane);
                        const double Sv = inc + S;
                        S += __shfl_sync(kFullMask, inc, 31);
                        if (valid && i >= i0) {
                            if (Sv > 0.0) {
                                prod_add(i, hd * log(Sv));
                                row[i] = e / Sv;
                            } else {  // cmf == 0: prod = -inf, E = 0 (prob.rs:81-85)
                                prod_add(i, NEG_INF);
                                row[i] = 0.0;
                            }
                        }
                    }
                    for (u32 i = i0 + lane; i < lo; i += 32) prod_add(i, NEG_INF);  // pmf underflows: cmf == 0 there
                    const double cf = hd * log(S);  // beyond hi the running sum no longer moves
                    for (u32 i = max(hi, i0) + lane; i <= t; i += 32) prod_add(i, cf);
                    if (lane == 0) {
                        sm.wlo[d] = (u16)max(lo, i0);
                        sm.whi[d] = (u16)hi;
                    }
                }
                __syncwarp();
            }
            __syncthreads();
            // E(i) = exp(prod(i)); exp(-inf) = 0 reproduces the reference's `prod == -inf => 0` branch
            for (u32 i = tid; i <= t; i += kProbThreads) {
                double s = NEG_INF;
                if (i >= i0) {
                    s = 0.0;
#pragma unroll
                    for (int w = 0; w < kProbWarps; ++w)
                        if (w < sc.nprod) s += sm.prodw[(size_t)w * T1 + i];
                }
                sm.E[i] = exp(s);
            }
            __syncthreads();
            // ---- pass 2: P(m) = sum_i (pmf_m(i)/cmf_m(i)) * E(i)   (prob.rs:74-90), same warp as pass 1 ----------
            for (int d = (int)D - 1 - warp; d >= 0; d -= kProbWarps) {
                const u32 m = sm.dm[d];
                double val;
                if (m == 0) {
                    val = sm.E[0];  // p = [0,-inf,..], c = 0
                } else {
                    double s = 0.0;
                    const double* __restrict__ row = cbuf + (size_t)d * sc.tstride;
                    const u32 a = sm.wlo[d], e = sm.whi[d];
                    for (u32 i = a + lane; i < e; i += 32) s = fma(row[i], sm.E[i], s);
                    val = warp_sum(s);
                }
                if (lane == 0) sm.Pd[d] = val;
            }
        }
        __syncthreads();
        // ---- normalise (prob.rs:97-102) and global signal (lineage.rs:86-90) ---------------------------
        double sl = 0.0;
        for (u32 d = tid; d < D; d += kProbThreads) sl += (double)sm.dh[d] * sm.Pd[d];
        const double S = block_sum(sl, red, tid, kProbWarps);
        const bool bad_sum = !(S > 0.0);  // assert!(probs_sum > 0.0)
        double gl = 0.0;
        for (u32 d = tid; d < D; d += kProbThreads) {
            double pn = sm.Pd[d] / S;
            ptab[sm.dm[d]] = pn;
            double df = pn - 1.0 / Nd;
            gl += (double)sm.dh[d] * (df * df);
        }
        const double gsum = block_sum(gl, red, tid, kProbWarps);
        if (tid == 0) {
            pool.global_sig[q] = sqrt(gsum);
            pool.status[q] = bad_sum ? kQProbSumZero : kQOk;
        }
        // m_min: the references whose count lies below it hold, all together, no more than kMassCut of the probability mass
        // (the histogram tells without touching the count vector); K4 takes them as exactly 0 -- 1e-9 of the 1.1e-16 rounding
        // noise the reference's own sequential prefix sums carry (lineage.rs:66-71)
        if (warp == 0) {
            double run = 0.0;
            u32 mmin = 0;  // 0 keeps every reference (also the answer when the sum is not a number)
            if (!bad_sum) {
                for (u32 base = 0; base < D; base += 32) {
                    const u32 d = base + lane;
                    const double v = d < D ? (double)sm.dh[d] * (sm.Pd[d] / S) : 0.0;
                    const double inc = warp_scan_incl(v, lane) + run;
                    const u32 hit = __ballot_sync(kFullMask, d < D && inc > kMassCut);
                    if (hit) {
                        mmin = sm.dm[base + (u32)__ffs(hit) - 1u];
                        break;
                    }
                    run = __shfl_sync(kFullMask, inc, 31);
                }
            }
            if (lane == 0) const_cast<u32*>(seg_aux(sc, ql))[0] = mmin;
        }
    }
}

// =========================================================================================================
// K4: prefix sums of the normalised probabilities (lineage.rs:61-77,114-117), kept per block of 8 references.
//
// One CTA per query, ONE barrier-free pass over the count vector in 512-reference segments (one segment = one warp
// iteration, 16 references per lane): thread-serial + warp scan of P(count[r]); the running sum at the start of every block of 8
// references -- two per lane, relative to the segment start -- is stored (64 values, 512 bytes per segment; round 1 stored the
// value at every node boundary, ~2.9 KB per segment on 1 M references, which made this kernel HBM-write-bound on flat profiles:
// 12.1 -> 6.2 ms per 20 k queries), the segment total goes to shared memory.  After the pass one block-wide exclusive scan turns the
// totals into segment offsets (a few KB per query).  The mass in front of a reference is then segoff[segment] + blk[block] + the up
// to 8 values P(count[r]) in between (mass_rel: one 16-byte load of the block's counts), and a node confidence
//     (segoff[seg(hi)] - segoff[seg(lo)]) + (rel(hi) - rel(lo))                                        (node_conf)
// -- or, for a node of at most 4 references, the sum of their probabilities themselves.  No warp ever waits for another one and the
// P(m) table is gathered exactly once per reference here.
// dynamic smem: double Ptab[hstride] | double segtot[n_seg (even)] | u32 skip bitmap words
// =========================================================================================================
constexpr int kPrefixThreads = 256;
constexpr int kPrefixWarps = kPrefixThreads / 32;
constexpr int kPrefixPer = 16;
constexpr u32 kPrefixSeg = 32 * kPrefixPer;  // 512 references; n_pad (a multiple of 4096) is a whole number of segments
static_assert(kPrefixSeg == 512, "node_conf / mass_rel shift by 9");

__device__ __forceinline__ void prefix_gather(double (&v)[kPrefixPer], const double* __restrict__ Ptab, const uint4& c0, const uint4& c1,
                                              u64 r0, u64 Ns) {
    const u32 w[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
    if (r0 + kPrefixPer <= Ns) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[2 * k] = Ptab[w[k] & 0xFFFFu];
            v[2 * k + 1] = Ptab[w[k] >> 16];
        }
    } else {  // padding references beyond the shard carry no probability
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[2 * k] = (r0 + 2 * k < Ns) ? Ptab[w[k] & 0xFFFFu] : 0.0;
            v[2 * k + 1] = (r0 + 2 * k + 1 < Ns) ? Ptab[w[k] >> 16] : 0.0;
        }
    }
}

__global__ void __launch_bounds__(kPrefixThreads)
    prefix_kernel(IndexView ix, BatchView b, ProbScratch sc, const u16* __restrict__ counts, int q_base, int q_count, int use_segmax) {
    extern __shared__ __align__(16) unsigned char xsm_raw[];
    __shared__ double wtot[kPrefixWarps];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ql = blockIdx.x;
    if (ql >= q_count) return;
    const int q = q_base + ql;
    const u32 n_seg = (u32)(ix.n_pad / kPrefixSeg);
    const bool ptab_global = sc.big != nullptr;  // very long queries: P(m) is gathered from the global table (L2) instead of a shared-memory copy
    double* segtot = reinterpret_cast<double*>(xsm_raw) + (ptab_global ? 0u : b.hstride);
    double* stage_end = segtot + ((n_seg + 1u) & ~1u);  // u32 skip bitmap words behind the segment totals
    const u32 K = b.K[q];
    const double* __restrict__ gp = sc.ptab + (size_t)ql * b.hstride;
    const double* __restrict__ Ptab = gp;
    if (!ptab_global) {
        double* Ps = reinterpret_cast<double*>(xsm_raw);
        for (u32 m = tid; m <= K; m += kPrefixThreads) Ps[m] = gp[m];
        Ptab = Ps;
    }
    __syncthreads();
    const u16* __restrict__ qcounts = counts + (size_t)ql * ix.n_pad;
    double* __restrict__ blk = sc.blk + (size_t)ql * sc.blk_stride;
    const u64 Ns = ix.shard_refs;
    u32* __restrict__ aux = const_cast<u32*>(seg_aux(sc, ql));
    const u32 mmin2 = aux[0] * 0x10001u;  // m_min in both half-words
    // per-segment maxima left by the hit-count kernel (upper bounds in skip mode, where exact matches were zeroed afterwards)
    const u16* __restrict__ smax = use_segmax ? seg_max(sc, ql, n_seg) : nullptr;
    u32* skipw_s = reinterpret_cast<u32*>(stage_end);
    for (u32 i = tid; i < (n_seg + 31u) / 32u; i += kPrefixThreads) skipw_s[i] = 0u;
    __syncthreads();

    const u32 mmin = aux[0];
    // a segment whose maximum stays below m_min is dropped without its counts ever being requested
    auto dropped = [&](u32 s) { return smax != nullptr && (u32)smax[s] < mmin; };
    uint4 c0 = make_uint4(0, 0, 0, 0), c1 = c0;
    if ((u32)warp < n_seg && !dropped(warp)) {
        const u64 r0 = (u64)warp * kPrefixSeg + (u64)lane * kPrefixPer;
        c0 = *reinterpret_cast<const uint4*>(qcounts + r0);
        c1 = *reinterpret_cast<const uint4*>(qcounts + r0 + 8);
    }
    for (u32 s = warp; s < n_seg; s += kPrefixWarps) {
        const u64 r0 = (u64)s * kPrefixSeg + (u64)lane * kPrefixPer;
        const uint4 x0 = c0, x1 = c1;
        const bool drop_this = dropped(s);
        if (s + kPrefixWarps < n_seg && !dropped(s + kPrefixWarps)) {  // the next segment's counts are requested before this one is used
            const u64 rn = r0 + (u64)kPrefixWarps * kPrefixSeg;
            c0 = *reinterpret_cast<const uint4*>(qcounts + rn);
            c1 = *reinterpret_cast<const uint4*>(qcounts + rn + 8);
        }
        if (drop_this) {
            if (lane == 0) {
                segtot[s] = 0.0;
                atomicOr(&skipw_s[s >> 5], 1u << (s & 31));
            }
            continue;
        }
        {   // does any reference of the segment reach m_min?  (padding references have count 0; m_min == 0 keeps everything)
            const u32 mx = __vmaxu2(__vmaxu2(__vmaxu2(x0.x, x0.y), __vmaxu2(x0.z, x0.w)), __vmaxu2(__vmaxu2(x1.x, x1.y), __vmaxu2(x1.z, x1.w)));
            if (!__any_sync(kFullMask, __vcmpgeu2(mx, mmin2) != 0u)) {
                if (lane == 0) {
                    segtot[s] = 0.0;
                    atomicOr(&skipw_s[s >> 5], 1u << (s & 31));
                }
                continue;
            }
        }
        double v[kPrefixPer];
        prefix_gather(v, Ptab, x0, x1, r0, Ns);
#pragma unroll
        for (int k = 1; k < kPrefixPer; ++k) v[k] += v[k - 1];
        const double inc = warp_scan_incl(v[kPrefixPer - 1], lane);
        const double offs = inc - v[kPrefixPer - 1];
        if (lane == 31) segtot[s] = inc;
        // the running sum at the start of every block of 8 references (two per lane), relative to the segment start
        *reinterpret_cast<double2*>(blk + (size_t)s * (kPrefixSeg / kBlkRefs) + 2 * lane) = make_double2(offs, offs + v[7]);
    }
    __syncthreads();
    // ---- exclusive scan of the segment totals -> segment offsets -------------------------------------------------
    {
        double* __restrict__ gseg = sc.segoff + (size_t)ql * sc.segoff_stride;
        const u32 per = (n_seg + kPrefixThreads - 1) / kPrefixThreads;
        const u32 lo = min(n_seg, (u32)tid * per), hi = min(n_seg, lo + per);
        double loc = 0.0;
        for (u32 i = lo; i < hi; ++i) loc += segtot[i];
        const double inc = warp_scan_incl(loc, lane);
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        double run = inc - loc;
#pragma unroll
        for (int w2 = 0; w2 < kPrefixWarps; ++w2)
            if (w2 < warp) run += wtot[w2];
        for (u32 i = lo; i < hi; ++i) {
            gseg[i] = run;
            run += segtot[i];
        }
    }
    for (u32 i = tid; i < (n_seg + 31u) / 32u; i += kPrefixThreads) aux[2 + i] = skipw_s[i];
}

// =========================================================================================================
// Best hits (RTX_OPT_BEST_HITS = T): the references with count >= 1, by count descending then id ascending, first min(T, #) of
// them.  One CTA per query of the sub-batch, behind the skip zeroing and the strand decision, while the count row is resident.
//   1. From the histogram, scanning down from K: tau = the largest m >= 1 with #{c >= m} >= T (1 if fewer than T references have a
//      hit) and g = #{c > tau} < T.  Exactly the g references above tau and the T - g lowest ids at tau are wanted.
//   2. Candidate segments (512 references): those whose maximum reaches tau, every one when there are no per-segment maxima.  In skip
//      mode the maxima were taken before the zeroing and are only upper bounds: they filter, nothing more.
//   3. The candidates in ascending id order, one warp per segment: every count > tau and the first ties at tau, positions from a
//      block-ordered prefix.  The histogram is exact, so the scan stops once both targets are met.
//   4. The < T counts above tau ranked by (count desc, id asc), the ties behind them in id order.
// =========================================================================================================
constexpr int kBestThreads = 256;
constexpr int kBestWarps = kBestThreads / 32;
constexpr u32 kBestHitsMax = 64;

__global__ void __launch_bounds__(kBestThreads)
    best_hits_kernel(IndexView ix, BatchView b, ProbScratch sc, const u16* __restrict__ counts, int use_segmax, u32 T, int q_base,
                     u32* __restrict__ n_hits, u32* __restrict__ hit_ref, u16* __restrict__ hit_count) {
    __shared__ u32 wsum[kBestWarps];
    __shared__ u32 s_tau, s_g;
    __shared__ u32 s_cand[kBestThreads];
    __shared__ u32 s_above_ref[kBestHitsMax], s_tie_ref[kBestHitsMax];
    __shared__ u16 s_above_cnt[kBestHitsMax];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ql = blockIdx.x, q = q_base + ql;
    const u32 K = b.K[q];
    const u32* __restrict__ hist = b.hist + (size_t)q * b.hstride;
    if (tid == 0) s_tau = 0;
    __syncthreads();
    // ---- 1. threshold: thread t of a round holds bucket top - t; its exclusive prefix is #{c > m} ------------------------------
    u32 above = 0;  // #{c > the round's lowest bucket}
    for (u32 top = K; top > 0; top -= min(top, (u32)kBestThreads)) {
        const u32 m = top - (u32)tid;
        const u32 h = (u32)tid < top ? hist[m] : 0u;
        u32 total;
        const u32 gt = above + block_scan_excl(h, wsum, tid, kBestWarps, &total);
        if (h && gt < T && gt + h >= T) {  // the one bucket where #{c >= m} reaches T
            s_tau = m;
            s_g = gt;
        }
        __syncthreads();
        if (s_tau) break;
        above += total;
    }
    u32 tau = s_tau, g = s_g;
    if (tau == 0) {  // fewer than T references with a hit: all of them
        tau = 1;
        g = K >= 1 ? above - hist[1] : 0u;
    }
    const u32 with_hit = K >= 1 ? (s_tau ? T : above) : 0u;
    const u32 need_tie = with_hit - g;
    if (with_hit == 0) {
        if (tid == 0) n_hits[q] = 0;
        return;
    }
    // ---- 2./3. candidate segments in windows of kBestThreads, then one warp per candidate ----------------------------------------
    const u32 Ns = (u32)ix.shard_refs;
    const u32 n_seg = (u32)(ix.n_pad / kPrefixSeg), n_seg_refs = (Ns + kPrefixSeg - 1) / kPrefixSeg;
    const u16* __restrict__ smax = use_segmax ? seg_max(sc, ql, n_seg) : nullptr;
    const u16* __restrict__ row = counts + (size_t)ql * ix.n_pad;
    u32 got_above = 0, got_tie = 0;
    bool done = false;
    for (u32 w0 = 0; w0 < n_seg_refs && !done; w0 += kBestThreads) {
        const u32 s = w0 + (u32)tid;
        const u32 cand = s < n_seg_refs && (smax == nullptr || (u32)smax[s] >= tau) ? 1u : 0u;
        u32 n_cand;
        const u32 slot = block_scan_excl(cand, wsum, tid, kBestWarps, &n_cand);
        if (cand) s_cand[slot] = s;
        __syncthreads();
        for (u32 c0 = 0; c0 < n_cand; c0 += kBestWarps) {
            const u32 ci = c0 + (u32)warp;
            u32 r0 = Ns;  // no segment for this warp: every reference reads as past the end
            uint4 x0 = make_uint4(0, 0, 0, 0), x1 = x0;
            if (ci < n_cand) {
                r0 = s_cand[ci] * kPrefixSeg + (u32)lane * 16u;
                x0 = *reinterpret_cast<const uint4*>(row + r0);
                x1 = *reinterpret_cast<const uint4*>(row + r0 + 8);
            }
            const u32 w[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
            u32 n_above = 0, n_tie = 0;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const u32 c = r0 + (u32)i < Ns ? (w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu : 0u;
                n_above += c > tau;
                n_tie += c == tau;
            }
            u32 total;  // both counts packed: at most kBestThreads * 16 per round
            const u32 ex = block_scan_excl(n_above | n_tie << 16, wsum, tid, kBestWarps, &total);
            u32 pa = got_above + (ex & 0xFFFFu), pt = got_tie + (ex >> 16);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const u32 c = r0 + (u32)i < Ns ? (w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu : 0u;
                if (c > tau) {
                    if (pa < kBestHitsMax) {
                        s_above_ref[pa] = r0 + (u32)i;
                        s_above_cnt[pa] = (u16)c;
                    }
                    ++pa;
                } else if (c == tau) {
                    if (pt < need_tie) s_tie_ref[pt] = r0 + (u32)i;
                    ++pt;
                }
            }
            got_above += total & 0xFFFFu;
            got_tie += total >> 16;
            if (got_above >= g && got_tie >= need_tie) {
                done = true;
                break;
            }
        }
    }
    __syncthreads();
    // ---- 4. rank the counts above tau; the ties follow in id order -------------------------------------------------------------
    u32* __restrict__ out_ref = hit_ref + (size_t)q * T;
    u16* __restrict__ out_cnt = hit_count + (size_t)q * T;
    const u64 id0 = ix.shard_begin;
    if ((u32)tid < g) {
        const u32 c = s_above_cnt[tid], r = s_above_ref[tid];
        u32 rank = 0;
        for (u32 j = 0; j < g; ++j) {
            const u32 cj = s_above_cnt[j];
            rank += cj > c || (cj == c && s_above_ref[j] < r);
        }
        out_ref[rank] = (u32)(id0 + r);
        out_cnt[rank] = (u16)c;
    }
    if ((u32)tid < need_tie) {
        out_ref[g + tid] = (u32)(id0 + s_tie_ref[tid]);
        out_cnt[g + tid] = (u16)tau;
    }
    if (tid == 0) n_hits[q] = with_hit;
}

// =========================================================================================================
// Reference-sharded mode.  A node whose reference range crosses a shard cut ("straddler") cannot be evaluated by one
// rank: every rank contributes a record per (query, straddler) -- its local probability mass, and what it knows about
// the straddler's children that lie wholly inside its shard -- the records are all-gathered, and each rank then walks
// the part of the tree it owns with the combined values.
// =========================================================================================================
struct ShardRec {
    double mass;     // sum of normalised probabilities of the straddler's references inside this shard
    double best;     // largest confidence among the straddler's non-straddling children inside this shard (-inf if none)
    u32 best_child;  // node id of the last such child within 1e-12 relative of `best`
    u32 n_sig;       // low half: how many of those children have round(conf*100) != 0; high half: below how many of them a line is pushed
};

struct ShardView {
    u32 n_strad, n_shards, rank, pad;
    const int* strad_of_node;  // [n_nodes] straddler index or -1
    const u32* strad_nodes;    // [n_strad]
    const int* strad_parent;   // [n_strad] straddler index of the parent node or -1
    ShardRec* send;            // [Q][n_strad]
    const ShardRec* recv;      // [n_shards][Q][n_strad]
    u8* sk;                    // [Q][n_strad] combined round(conf*100)
    u8* sany;                  // [Q][n_strad] combined: bit 0 "has a significant child" (Inner: fallback or not), bit 1 "a line is pushed below" (Taxon: report or not)
    u32* sbest;                // [Q][n_strad] combined best child (node id)
};

__device__ __forceinline__ bool node_inside(const IndexView& ix, u32 node) {
    return ix.node_lo[node] >= ix.shard_begin && ix.node_hi[node] <= ix.shard_begin + ix.shard_refs;
}

// Does the subtree of a significant Sequence node push a result line (lineage.rs:126-149)?  Its Taxon / Inner children do as soon as
// they are significant; Sequence children (a rank repeating its parent's label again) are followed.  The node lies inside the shard,
// hence so does its whole subtree.  Rare path (degenerate lineages), one lane.
__device__ bool seq_subtree_pushes(const NodeRec* __restrict__ recs, const MassView& mv, const NodeRec& s) {
    u32 st_cf[8], st_cc[8];
    int sp = 1;
    st_cf[0] = s.child_first;
    st_cc[0] = s.cc_type & 0x3FFFFFFFu;
    while (sp > 0) {
        --sp;
        const u32 cf = st_cf[sp], cc = st_cc[sp];
        for (u32 i = 0; i < cc; ++i) {
            const NodeRec c = recs[cf + i];
            if ((u32)round(node_conf(mv, c) * 100.0) == 0u) continue;
            if ((c.cc_type >> 30) != 2u) return true;
            if (sp >= 8) return true;  // deeper than any sane lineage: be conservative
            st_cf[sp] = c.child_first;
            st_cc[sp] = c.cc_type & 0x3FFFFFFFu;
            ++sp;
        }
    }
    return false;
}

// One warp per (query, straddler): the straddler's probability mass inside this shard and, of its children that lie wholly inside the
// shard, how many are significant / push a line and which one is the largest (last one within 1e-12 relative of the maximum, as in
// lineage.rs:156-164; the ranks' records are combined by shard_combine_kernel).
//   * Only the children that touch the shard are looked at (binary search over the sorted child ranges).
//   * One pass: the last "record" (a child within the tolerance of the running maximum) is the answer if it passes the final test, see
//     the fallback rounds of lineage_bfs_kernel; else the run is scanned again.
//   * A query that kept few 512-reference segments under the straddler (K4's mass cut) only evaluates the children that overlap
//     them; all others are exactly 0 -- they only matter when nothing is above 0, and then the last child wins.
constexpr u32 kRecKept = 32;        // at most this many kept segments under a straddler for the sparse scan
constexpr u32 kRecSparseMin = 128;  // children touching the shard, below which everything is evaluated

__global__ void __launch_bounds__(128) shard_records_kernel(IndexView ix, const NodeRec* __restrict__ recs, ProbScratch sc, ShardView sv, int q_count) {
    __shared__ u32 s_kept[4][kRecKept];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= (long long)q_count * sv.n_strad) return;
    const int ql = (int)(w / sv.n_strad), j = (int)(w % sv.n_strad);
    const MassView mv = mass_view(sc, ql);
    const u64 sh_lo = ix.shard_begin, sh_hi = ix.shard_begin + ix.shard_refs;
    const u32 node = sv.strad_nodes[j];
    const NodeRec nr = recs[node];
    const u32 cf = nr.child_first, cc = nr.cc_type & 0x3FFFFFFFu;
    auto child_lo_size = [&](u32 ci) { return *reinterpret_cast<const uint2*>(&recs[cf + ci].lo); };
    // children [ta, tb) touch the shard
    u32 ta = 0, tb = cc;
    if (cc > 32) {
        ta = warp_first_true(0u, cc, lane, [&](u32 x) { const uint2 ls = child_lo_size(x); return (u64)ls.x + ls.y > sh_lo; });
        tb = warp_first_true(ta, cc, lane, [&](u32 x) { return (u64)child_lo_size(x).x >= sh_hi; });
    }
    double best = -CUDART_INF;
    u32 n_sig = 0, n_push = 0;  // significant inside children; those of them below which a result line is pushed (per lane)
    u32 last_rec = 0, last_valid = 0;  // 1 + child index (warp-uniform)
    auto conf_of = [&](u32 ci, bool& valid) {
        const NodeRec cr = recs[cf + ci];
        valid = sv.strad_of_node[cf + ci] < 0 && (u64)cr.lo >= sh_lo && (u64)cr.lo + cr.size <= sh_hi;
        return cr;
    };
    auto scan_run = [&](u32 a, u32 b2) {
        for (u32 cb = a; cb < b2; cb += 32) {
            const u32 ci = cb + lane;
            bool valid = false;
            double v = -CUDART_INF;
            if (ci < b2) {
                const NodeRec cr = conf_of(ci, valid);
                if (valid) {
                    v = node_conf(mv, cr);
                    if ((u32)round(v * 100.0) != 0) {
                        ++n_sig;
                        n_push += ((cr.cc_type >> 30) != 2u) || seq_subtree_pushes(recs, mv, cr);
                    }
                }
            }
            const u32 vm = __ballot_sync(kFullMask, valid);
            if (vm == 0u) continue;
            double vmax = v;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(kFullMask, vmax, o));
            best = fmax(best, vmax);
            const bool rec = valid && v >= best - fabs(best) * 1e-12;
            const u32 r = __reduce_max_sync(kFullMask, rec ? ci + 1u : 0u);
            if (r) last_rec = r;
            last_valid = cb + 32u - (u32)__clz(vm);  // 1 + index of the chunk's last valid child (chunks ascend)
        }
    };
    // the kept segments under the part of the straddler that lies in this shard
    bool sparse = false;
    u32 n_kept = 0;
    if (tb - ta > kRecSparseMin) {
        const u64 llo = (u64)nr.lo > sh_lo ? (u64)nr.lo - sh_lo : 0ull;
        const u64 lhi = min((u64)nr.lo + nr.size, sh_hi) - sh_lo;
        const u32 s0 = (u32)(llo / kPrefixSeg), s1 = (u32)((lhi + kPrefixSeg - 1) / kPrefixSeg);  // segments [s0, s1)
        sparse = true;
        for (u32 wb = s0 >> 5; wb * 32u < s1 && sparse; wb += 32) {
            const u32 wi = wb + lane;
            u32 kw = 0;
            if (wi * 32u < s1) {
                kw = ~mv.skipw[wi];
                if (wi * 32u < s0) kw &= ~((1u << (s0 - wi * 32u)) - 1u);
                if (wi * 32u + 32u > s1) kw &= (1u << (s1 - wi * 32u)) - 1u;
            }
            const u32 c = __popc(kw);
            const u32 inc = warp_scan_incl(c, lane);
            const u32 tot = __shfl_sync(kFullMask, inc, 31);
            if (n_kept + tot > kRecKept) {
                sparse = false;
            } else {
                u32 pos = n_kept + inc - c;
                while (kw) {
                    s_kept[wib][pos++] = wi * 32u + (u32)__ffs(kw) - 1u;
                    kw &= kw - 1u;
                }
                n_kept += tot;
            }
        }
        __syncwarp();
    }
    if (sparse) {
        u32 cursor = ta;
        for (u32 k = 0; k < n_kept && cursor < tb; ++k) {
            const u64 key_lo = sh_lo + (u64)s_kept[wib][k] * kPrefixSeg, key_hi = key_lo + kPrefixSeg;
            const u32 a = warp_first_true(cursor, tb, lane, [&](u32 x) { const uint2 ls = child_lo_size(x); return (u64)ls.x + ls.y > key_lo; });
            const u32 b2 = warp_first_true(a, tb, lane, [&](u32 x) { return (u64)child_lo_size(x).x >= key_hi; });
            scan_run(a, b2);
            cursor = max(cursor, b2);
        }
        if (!(best > 0.0)) {  // nothing above 0 among the evaluated children: the others are exactly 0, all tie, the last valid child wins
            bool v1 = false, v2 = false;
            if (tb > ta) conf_of(tb - 1, v1);
            if (tb > ta + 1) conf_of(tb - 2, v2);
            const u32 lv = v1 ? tb : (v2 ? tb - 1 : 0u);
            if (lv) {
                best = fmax(best, 0.0);
                last_rec = lv;
            }
            last_valid = 0;  // (no second pass)
        }
    } else {
        scan_run(ta, tb);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_sig += __shfl_xor_sync(kFullMask, n_sig, o);
        n_push += __shfl_xor_sync(kFullMask, n_push, o);
    }
    u32 besti = 0;
    if (best > -CUDART_INF && last_rec) {
        const double thr = best - fabs(best) * 1e-12;
        bool ok = true;
        if (last_valid) {  // does the last record pass the final test?
            bool valid;
            const NodeRec cr = conf_of(last_rec - 1u, valid);
            ok = node_conf(mv, cr) >= thr;
        }
        if (ok) {
            besti = cf + last_rec - 1u;
        } else {  // (values in the 1e-12 band right below the tolerance: practically never) second pass
            for (u32 cb = ta; cb < tb; cb += 32) {
                const u32 ci = cb + lane;
                if (ci < tb) {
                    bool valid;
                    const NodeRec cr = conf_of(ci, valid);
                    if (valid && node_conf(mv, cr) >= thr) besti = cf + ci;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) besti = max(besti, __shfl_xor_sync(kFullMask, besti, o));
        }
    }
    if (lane == 0) {
        ShardRec r;
        r.mass = node_conf(mv, nr);
        r.best = best;
        r.best_child = besti;
        r.n_sig = min(n_sig, 0xFFFFu) | (min(n_push, 0xFFFFu) << 16);
        sv.send[(size_t)ql * sv.n_strad + j] = r;
    }
}

// one thread per query: masses summed in rank order (deterministic), then any-significant-child and best child
__global__ void shard_combine_kernel(ShardView sv, const NodeRec* __restrict__ recs, int q_count) {
    const int ql = blockIdx.x * blockDim.x + threadIdx.x;
    if (ql >= q_count) return;
    const u32 S = sv.n_strad;
    const size_t rank_stride = (size_t)q_count * S;
    auto mass_of = [&](u32 j) {
        double m = 0.0;
        for (u32 r = 0; r < sv.n_shards; ++r) m += sv.recv[r * rank_stride + (size_t)ql * S + j].mass;
        return m;
    };
    for (u32 j = 0; j < S; ++j) sv.sk[(size_t)ql * S + j] = (u8)min((u32)round(mass_of(j) * 100.0), 255u);
    for (int j = (int)S - 1; j >= 0; --j) {  // children before parents (straddlers are listed in BFS order): spush of a child is final
        u32 nsig = 0, npush = 0;
        double gmax = -CUDART_INF;
        for (u32 r = 0; r < sv.n_shards; ++r) {
            const ShardRec rec = sv.recv[r * rank_stride + (size_t)ql * S + j];
            nsig += rec.n_sig & 0xFFFFu;
            npush += rec.n_sig >> 16;
            gmax = fmax(gmax, rec.best);
        }
        for (u32 c = 0; c < S; ++c)
            if (sv.strad_parent[c] == (int)j) {
                const bool sig = sv.sk[(size_t)ql * S + c] != 0;
                nsig += sig;
                // a significant straddling child pushes when it is a Taxon / Inner node, or a Sequence node below which something is pushed
                npush += sig && ((recs[sv.strad_nodes[c]].cc_type >> 30) != 2u || (sv.sany[(size_t)ql * S + c] & 2u));
                gmax = fmax(gmax, mass_of(c));
            }
        const double thr = gmax - fabs(gmax) * 1e-12;
        u32 best_child = 0;
        for (u32 r = 0; r < sv.n_shards; ++r) {
            const ShardRec rec = sv.recv[r * rank_stride + (size_t)ql * S + j];
            if (rec.best > -CUDART_INF && rec.best >= thr) best_child = max(best_child, rec.best_child);
        }
        for (u32 c = 0; c < S; ++c)
            if (sv.strad_parent[c] == (int)j && mass_of(c) >= thr) best_child = max(best_child, sv.strad_nodes[c]);
        sv.sany[(size_t)ql * S + j] = (u8)((nsig != 0) | ((npush != 0) << 1));  // bit 0: a significant child exists; bit 1: a line is pushed below
        sv.sbest[(size_t)ql * S + j] = best_child;
    }
}

// =========================================================================================================
// K5: tree walk, ordering, override, emission.  One warp per query (thousands of independent walkers hide the
// latency of the dependent loads); 4 warps per CTA.
//
// Lineage::eval_recurse (lineage.rs:119-179) as an explicit depth-first stack: a frame is (node, next child to
// look at, "had a significant child").  Confidences are carried as integers k = round(conf*100), so that the
// reported value k/100 is bit-identical to the reference's round(conf*100)/100.
// =========================================================================================================
constexpr int kWalkWarps = 1;  // one warp per CTA: a slot frees as soon as its walker finishes (2 per CTA measured equal: the tail is the longest walk)

// per-warp shared state; res_k rows have stride ML
struct WalkSmem {
    double* res_local;  // [R]
    u32* res_first;     // [R]
    u32* st_node;       // [RTX_MAX_LEVELS + 1]
    u32* st_next;
    u32* st_cf;         // child_first of the frame's node
    u32* st_cc;         // child_count | type << 30 of the frame's node
    u32* path_node;     // [RTX_MAX_LEVELS + 1]
    u16* order;         // [R]
    u8* res_nlev;       // [R]
    u8* res_k;          // [R][ML]
    u8* st_any;         // [RTX_MAX_LEVELS + 1]
    u8* path_k;         // [RTX_MAX_LEVELS + 1]
    static constexpr u32 R = RTX_MAX_RESULTS_PER_QUERY;
    static constexpr u32 L1 = RTX_MAX_LEVELS + 1;
    __host__ __device__ static size_t bytes(u32 ML) {
        size_t b = (size_t)R * (8 + 4 + 2 + 1 + ML) + (size_t)L1 * (4 * 5 + 2);
        return (b + 15) & ~(size_t)15;
    }
    __device__ WalkSmem(unsigned char* base, u32 ML) {
        res_local = reinterpret_cast<double*>(base);
        res_first = reinterpret_cast<u32*>(res_local + R);
        st_node = res_first + R;
        st_next = st_node + L1;
        st_cf = st_next + L1;
        st_cc = st_cf + L1;
        path_node = st_cc + L1;
        order = reinterpret_cast<u16*>(path_node + L1);
        res_nlev = reinterpret_cast<u8*>(order + R);
        res_k = res_nlev + R;
        st_any = res_k + (size_t)R * ML;
        path_k = st_any + L1;
    }
};

template <bool SH>
__global__ void __launch_bounds__(kWalkWarps * 32)
    lineage_walk_kernel(IndexView ix, const NodeRec* __restrict__ recs, BatchView b, ResultPool pool, ProbScratch sc, ShardView sv, int q_base,
                        int q_count, int retry_only) {
    extern __shared__ __align__(16) unsigned char wsm_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ql = blockIdx.x * kWalkWarps + warp;
    if (ql >= q_count) return;
    const int q = q_base + ql;
    if (retry_only) {  // clean-up pass behind lineage_bfs_kernel: only the queries whose significant-node log overflowed there
        if (pool.status[q] != kQWalkRetry) return;
        if (lane == 0) pool.status[q] = kQOk;
        __syncwarp();
    }
    const u32 ML = ix.max_levels;
    WalkSmem ws(wsm_raw + (size_t)warp * WalkSmem::bytes(ML), ML);
    const double Nd = (double)ix.n_refs;
    const MassView mv = mass_view(sc, ql);
    int status = retry_only ? (int)kQOk : pool.status[q];

    u32 n_res = 0;
    bool overflow = false;
    if (status == kQOk) {
        int depth = 0;
        if (lane == 0) {
            const NodeRec root = recs[0];
            ws.st_node[0] = 0;
            ws.st_next[0] = 0;
            ws.st_any[0] = 0;
            ws.st_cf[0] = root.child_first;
            ws.st_cc[0] = root.cc_type;
        }
        __syncwarp();
        while (depth >= 0) {
            const u32 node = ws.st_node[depth];
            const u32 cf = ws.st_cf[depth], cct = ws.st_cc[depth];
            const u32 cc = cct & 0x3FFFFFFFu, ntype = cct >> 30;
            u32 nxt = ws.st_next[depth];
            bool found = false;
            u32 child = 0, ck = 0, ccf = 0, ccc = 0;
            for (u32 cb = nxt; cb < cc; cb += 32) {
                const u32 ci = cb + lane;
                u32 k = 0;
                NodeRec cr = NodeRec{0, 0, 0, 0, 0, 0, 0, 0};
                if (ci < cc) {
                    cr = recs[cf + ci];
                    if (SH) {
                        const int sj = sv.strad_of_node[cf + ci];
                        if (sj >= 0) k = sv.sk[(size_t)ql * sv.n_strad + sj];  // combined over the ranks
                        else if (node_inside(ix, cf + ci)) k = (u32)round((node_conf(mv, cr)) * 100.0);
                        // children inside another shard are walked by their owner
                    } else {
                        k = (u32)round((node_conf(mv, cr)) * 100.0);  // f64::round, half away from zero (lineage.rs:129)
                    }
                }
                const u32 mask = __ballot_sync(kFullMask, k != 0);
                if (mask) {
                    const int j = __ffs(mask) - 1;
                    child = cf + cb + j;
                    ck = __shfl_sync(kFullMask, k, j);
                    ccf = __shfl_sync(kFullMask, cr.child_first, j);
                    ccc = __shfl_sync(kFullMask, cr.cc_type, j);
                    nxt = cb + j + 1;
                    found = true;
                    break;
                }
            }
            if (found) {
                if (depth >= RTX_MAX_LEVELS) {
                    overflow = true;
                    break;
                }
                __syncwarp();  // every lane has read this frame (top of the iteration) before lane 0 rewrites it
                if (lane == 0) {
                    ws.st_next[depth] = nxt;
                    ws.st_any[depth] |= 1;  // bit 0: a significant child exists; bit 1: something was pushed below (set on the way up)
                    ws.path_node[depth] = child;
                    ws.path_k[depth] = (u8)min(ck, 255u);
                    ws.st_node[depth + 1] = child;
                    ws.st_next[depth + 1] = 0;
                    ws.st_any[depth + 1] = 0;
                    ws.st_cf[depth + 1] = ccf;
                    ws.st_cc[depth + 1] = ccc;
                }
                __syncwarp();
                ++depth;
                continue;
            }
            // children exhausted.  lineage.rs:126-177 keeps two facts apart: an Inner node falls back when NO CHILD IS SIGNIFICANT, a
            // Taxon is reported by its parent when its recursion PUSHED NOTHING.  They differ only below a Taxon whose significant
            // child is a Sequence node that itself has children (a rank repeating its parent's label, tree.rs:77-107): such a
            // child is significant yet may push nothing.
            const u32 fl = ws.st_any[depth];
            bool any_sig = (fl & 1u) != 0, pushed = (fl & 2u) != 0;
            bool mine = true;  // does this rank emit for `node`?
            if (SH) {
                const int sj = sv.strad_of_node[node];
                if (sj >= 0) {
                    const u32 sa = sv.sany[(size_t)ql * sv.n_strad + sj];
                    any_sig = any_sig || (sa & 1u);
                    pushed = pushed || (sa & 2u);
                    mine = ix.node_lo[node] >= ix.shard_begin && ix.node_lo[node] < ix.shard_begin + ix.shard_refs;
                }
            }
            const bool emits = ntype == 0 ? !any_sig : (ntype == 1 && !pushed && depth != 0);  // by this rank or the owner of the node
            pushed = pushed || emits;
            if (emits && (ntype == 0 || mine)) {
                int d = depth;
                u32 cur = node;
                if (ntype == 0) {  // Inner without a significant child: follow the best children (lineage.rs:151-177)
                    u32 cur_cf = cf, cur_cc = cc, cur_type = 0;
                    while (cur_type == 0 && d < RTX_MAX_LEVELS) {
                        if (SH) {
                            const int sj = sv.strad_of_node[cur];
                            if (sj >= 0) {  // the best child of a straddler was decided from all ranks' records
                                cur = sv.sbest[(size_t)ql * sv.n_strad + sj];
                                const NodeRec br = recs[cur];
                                if (lane == 0) {
                                    ws.path_node[d] = cur;
                                    ws.path_k[d] = 1;
                                }
                                ++d;
                                cur_cf = br.child_first;
                                cur_cc = br.cc_type & 0x3FFFFFFFu;
                                cur_type = br.cc_type >> 30;
                                continue;
                            }
                            if (!node_inside(ix, cur)) break;  // the chain continues in another rank's shard
                        }
                        // max_by(partial_cmp): the LAST maximal child wins (lineage.rs:156-164).  Children tied in exact
                        // arithmetic (same hit counts) differ here only by rounding noise of the prefix sums, so values
                        // within 1e-12 relative of the maximum count as maximal.
                        double best = -CUDART_INF;
                        double cv0 = -CUDART_INF;      // this lane's child of the first 32 (kept for the second pass)
                        NodeRec cr0 = NodeRec{0, 0, 0, 0, 0, 0, 0, 0};
                        for (u32 cb = 0; cb < cur_cc; cb += 32) {
                            const u32 ci = cb + lane;
                            if (ci < cur_cc) {
                                const NodeRec cr = recs[cur_cf + ci];
                                const double v = node_conf(mv, cr);
                                if (cb == 0) {
                                    cv0 = v;
                                    cr0 = cr;
                                }
                                best = fmax(best, v);
                            }
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(kFullMask, best, o));
                        const double thr = best - fabs(best) * 1e-12;
                        u32 besti = 0;
                        if (lane < cur_cc && cv0 >= thr) besti = lane;
                        for (u32 cb = 32; cb < cur_cc; cb += 32) {
                            const u32 ci = cb + lane;
                            if (ci < cur_cc) {
                                const NodeRec cr = recs[cur_cf + ci];
                                if (node_conf(mv, cr) >= thr) besti = ci;
                            }
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) besti = max(besti, __shfl_xor_sync(kFullMask, besti, o));
                        cur = cur_cf + besti;
                        NodeRec br;
                        if (besti < 32) {  // the winner's record is already in a register of lane besti
                            br.child_first = __shfl_sync(kFullMask, cr0.child_first, besti);
                            br.cc_type = __shfl_sync(kFullMask, cr0.cc_type, besti);
                        } else {
                            br = recs[cur];
                        }
                        if (lane == 0) {
                            ws.path_node[d] = cur;
                            ws.path_k[d] = 1;  // 1.0 / rounding_factor
                        }
                        ++d;
                        cur_cf = br.child_first;
                        cur_cc = br.cc_type & 0x3FFFFFFFu;
                        cur_type = br.cc_type >> 30;
                    }
                    if (SH) {
                        const int sj = sv.strad_of_node[cur];
                        mine = cur_type != 0 && (sj >= 0 ? (ix.node_lo[cur] >= ix.shard_begin && ix.node_lo[cur] < ix.shard_begin + ix.shard_refs)
                                                         : node_inside(ix, cur));
                    } else if (cur_type == 0) overflow = true;
                }
                __syncwarp();
                if (mine && n_res >= RTX_MAX_RESULTS_PER_QUERY) overflow = true;
                if (mine && !overflow) {
                    // confidence / expected vectors of this line; local signal (lineage.rs:95-102, utils.rs:91-105)
                    double cv = 0.0, ev = 0.0;
                    if (lane < d) {
                        const u32 nd = ws.path_node[lane];
                        cv = (double)ws.path_k[lane] / 100.0;
                        ev = (double)(ix.node_hi[nd] - ix.node_lo[nd]) / Nd;
                        ws.res_k[(size_t)n_res * ML + lane] = ws.path_k[lane];
                    }
                    const u32 lt1 = __ballot_sync(kFullMask, lane < d && 1.0 > ev);
                    const int start = lt1 ? (__ffs(lt1) - 1) : (d - 1);
                    double a_sum = 0.0, b_sum = 0.0;  // sequential sums, level order, like the reference
                    for (int i2 = start; i2 < d; ++i2) {
                        a_sum += __shfl_sync(kFullMask, cv, i2);
                        b_sum += __shfl_sync(kFullMask, ev, i2);
                    }
                    double s2 = 0.0;
                    for (int i2 = start; i2 < d; ++i2) {
                        const double df = __shfl_sync(kFullMask, cv, i2) / a_sum - __shfl_sync(kFullMask, ev, i2) / b_sum;
                        s2 += df * df;
                    }
                    if (lane == 0) {
                        ws.res_local[n_res] = sqrt(s2);
                        ws.res_first[n_res] = ix.node_lo[cur];
                        ws.res_nlev[n_res] = (u8)d;
                    }
                    ++n_res;
                }
                if (overflow) break;
            }
            --depth;
            if (depth >= 0 && pushed && lane == 0) ws.st_any[depth] |= 2;
            __syncwarp();
        }
        __syncwarp();
        if (overflow) status = kQTooManyResults;
        else if (n_res == 0 && !SH) status = kQEmptyResult;  // assert!(!eval_res.is_empty()) raxtax.rs:72 (sharded: checked after the merge)
    }
    // ---- order (lineage.rs:93): stable sort, descending lexicographic on the confidence vectors.  Results were pushed
    // in depth-first order, so the tie-break is the push index.
    if (status == kQOk) {
        for (u32 i = lane; i < n_res; i += 32) {
            const u8* ci = ws.res_k + (size_t)i * ML;
            const u32 li = ws.res_nlev[i];
            u32 rank = 0;
            for (u32 j = 0; j < n_res; ++j) {
                if (j == i) continue;
                const u8* cj = ws.res_k + (size_t)j * ML;
                const u32 lj = ws.res_nlev[j];
                int cmp = 0;  // +1: vector j > vector i
                for (u32 l = 0; l < min(li, lj); ++l) {
                    if (cj[l] != ci[l]) {
                        cmp = cj[l] > ci[l] ? 1 : -1;
                        break;
                    }
                }
                if (cmp == 0) cmp = (lj > li) ? 1 : (lj < li) ? -1 : 0;
                if (cmp > 0 || (cmp == 0 && j < i)) ++rank;
            }
            ws.order[rank] = (u16)i;
        }
    }
    __syncwarp();
    // ---- override (raxtax.rs:73-84) and emission into the result pool ---------------------------------------
    u32 n_out = (status == kQOk) ? n_res : 0;
    bool ovr = false;
    u32 ovr_idx = 0;
    if (!SH && status == kQOk && !(b.flags & RTX_RAW_CONFIDENCE) && !(b.flags & RTX_SKIP_EXACT_MATCHES) && b.exact_off) {
        if (b.exact_off[q + 1] - b.exact_off[q] == 1) {  // sharded: the caller applies the override after merging the ranks
            ovr = true;
            ovr_idx = b.exact_ids[b.exact_off[q]];
            n_out = 1;
        }
    }
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(pool.used, (unsigned long long)n_out);
    base = __shfl_sync(kFullMask, base, 0);
    if (base + n_out > pool.cap) {
        if (status == kQOk) status = kQPoolOverflow;
    } else if (ovr) {
        const u32 nl = ix.ref_levels[ovr_idx];
        if (lane == 0) {
            pool.first_ref[base] = ovr_idx;
            pool.n_levels[base] = (u8)nl;
            pool.local[base] = ws.res_local[ws.order[0]];
        }
        for (u32 l = lane; l < ML; l += 32) pool.conf[base * ML + l] = (l < nl) ? 1.0 : 0.0;
    } else {
        for (u32 x = lane; x < n_out * ML; x += 32) {
            const u32 i = x / ML, l = x - i * ML;
            const u32 src = ws.order[i];
            pool.conf[(base + i) * ML + l] = (l < ws.res_nlev[src]) ? (double)ws.res_k[(size_t)src * ML + l] / 100.0 : 0.0;
        }
        for (u32 i = lane; i < n_out; i += 32) {
            const u32 src = ws.order[i];
            pool.first_ref[base + i] = ws.res_first[src];
            pool.n_levels[base + i] = ws.res_nlev[src];
            pool.local[base + i] = ws.res_local[src];
        }
    }
    if (lane == 0) {
        pool.res_off[q] = (u32)base;
        pool.res_cnt[q] = n_out;
        pool.status[q] = status;
    }
}

// =========================================================================================================
// Result ordering.  The walk kernels append to the pool in completion order (one atomic bump per query); the two kernels
// below put the lines of a batch into query order on the device, so that the download is one contiguous copy per array
// and the host never touches individual results.
// =========================================================================================================
constexpr int kScanThreads = 1024;
// ord_begin[q] = sum of res_cnt[0..q), ord_begin[nq] = total.  Single CTA (nq <= a few 100 k: ~10 us).
__global__ void __launch_bounds__(kScanThreads) result_scan_kernel(ResultPool pool, u32* __restrict__ ord_begin, u32 nq) {
    __shared__ u32 wtot[kScanThreads / 32];
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 per = (nq + kScanThreads - 1) / kScanThreads;
    const u32 lo = min(nq, tid * per), hi = min(nq, lo + per);
    u32 loc = 0;
    for (u32 q = lo; q < hi; ++q) loc += pool.res_cnt[q];
    const u32 inc = warp_scan_incl(loc, (int)lane);
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const u32 v = wtot[lane];
        const u32 vi = warp_scan_incl(v, (int)lane);
        wtot[lane] = vi - v;
    }
    __syncthreads();
    u32 run = wtot[warp] + inc - loc;
    for (u32 q = lo; q < hi; ++q) {
        ord_begin[q] = run;
        run += pool.res_cnt[q];
    }
    if (tid == kScanThreads - 1) ord_begin[nq] = run;
}
// one warp per query; queries whose lines fell off the end of the pool (kQPoolOverflow: the batch is re-run) are left out
__global__ void __launch_bounds__(256) result_gather_kernel(ResultPool pool, const u32* __restrict__ ord_begin, u32* __restrict__ o_first,
                                                            u8* __restrict__ o_nlev, double* __restrict__ o_conf, double* __restrict__ o_local,
                                                            u32 nq, u32 ML) {
    const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= nq) return;
    const u64 src = pool.res_off[q], n = pool.res_cnt[q], dst = ord_begin[q];
    if (src + n > pool.cap || dst + n > pool.cap) return;
    for (u32 i = lane; i < n; i += 32) {
        o_first[dst + i] = pool.first_ref[src + i];
        o_nlev[dst + i] = pool.n_levels[src + i];
        o_local[dst + i] = pool.local[src + i];
    }
    for (u32 x = lane; x < n * ML; x += 32) o_conf[dst * ML + x] = pool.conf[src * ML + x];
}

// =========================================================================================================
// Reference-sharded mode, on the root after the result gather: per query the lines of ALL ranks -- each rank's already in the order of
// lineage.rs:93 -- merged into that order (confidence vectors descending lexicographically, on an equal prefix the longer vector
// first, then first reference ascending), followed by the one-exact-match override (raxtax.rs:73-84), which needs the best line of
// all ranks and is therefore left out by the ranks' own walks.  g_* hold the ranks' lines back to back (rank r at rank_off[r]),
// all_begin[r][q] the ranks' per-query offsets.
// =========================================================================================================
struct MergeView {
    const u32* all_begin;  // [n_ranks][nq + 1]
    const u32* rank_off;   // [n_ranks + 1] first line of rank r in g_*
    const u32* g_first;
    const u8* g_nlev;
    const double* g_conf;  // [lines][ML]
    const double* g_local;
    u32 n_ranks, nq, ML, pad;
};

__device__ __forceinline__ bool merge_override(const BatchView& b, u32 q) {
    if ((b.flags & (RTX_RAW_CONFIDENCE | RTX_SKIP_EXACT_MATCHES)) || b.exact_off == nullptr) return false;
    return b.exact_off[q + 1] - b.exact_off[q] == 1u;
}

// merged line count per query -> pool.res_cnt (result_scan_kernel then turns it into the offsets of the merged arrays)
__global__ void __launch_bounds__(256) shard_merge_count_kernel(MergeView mv, BatchView b, ResultPool pool) {
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= mv.nq) return;
    u32 tot = 0;
    for (u32 r = 0; r < mv.n_ranks; ++r) {
        const u32* ab = mv.all_begin + (size_t)r * (mv.nq + 1);
        tot += ab[q + 1] - ab[q];
    }
    if (tot == 0) pool.status[q] = kQEmptyResult;  // raxtax.rs:72
    else if (tot > RTX_MAX_RESULTS_PER_QUERY) pool.status[q] = kQTooManyResults;
    pool.res_cnt[q] = tot == 0 ? 0u : (merge_override(b, q) ? 1u : tot);
}

// one warp per query: rank sort of the query's lines (a handful; at most RTX_MAX_RESULTS_PER_QUERY)
__global__ void __launch_bounds__(256) shard_merge_write_kernel(MergeView mv, BatchView b, IndexView ix, const u32* __restrict__ ord_begin,
                                                                 u32* __restrict__ o_first, u8* __restrict__ o_nlev, double* __restrict__ o_conf,
                                                                 double* __restrict__ o_local) {
    const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= mv.nq) return;
    const u32 ML = mv.ML, R = mv.n_ranks;
    u32 tot = 0;
    for (u32 r = 0; r < R; ++r) {
        const u32* ab = mv.all_begin + (size_t)r * (mv.nq + 1);
        tot += ab[q + 1] - ab[q];
    }
    if (tot == 0 || tot > RTX_MAX_RESULTS_PER_QUERY) return;
    // i-th line of the query over the ranks in rank order -> index into g_*
    auto line_at = [&](u32 i) -> u32 {
        for (u32 r = 0; r < R; ++r) {
            const u32* ab = mv.all_begin + (size_t)r * (mv.nq + 1);
            const u32 n = ab[q + 1] - ab[q];
            if (i < n) return mv.rank_off[r] + ab[q] + i;
            i -= n;
        }
        return 0u;
    };
    // does line x come before line y?
    auto before = [&](u32 x, u32 y) -> bool {
        const u32 nx = mv.g_nlev[x], ny = mv.g_nlev[y];
        for (u32 lev = 0; lev < ML; ++lev) {
            const bool hx = lev < nx, hy = lev < ny;
            if (!hx && !hy) break;
            if (hx != hy) return hx;  // equal prefix: the longer vector first
            const long long kx = llround(mv.g_conf[(size_t)x * ML + lev] * 100.0), ky = llround(mv.g_conf[(size_t)y * ML + lev] * 100.0);
            if (kx != ky) return kx > ky;
        }
        const u32 fx = mv.g_first[x], fy = mv.g_first[y];
        return fx != fy ? fx < fy : x < y;
    };
    const bool ovr = merge_override(b, q);
    const u32 dst = ord_begin[q];
    for (u32 i = lane; i < tot; i += 32) {
        const u32 x = line_at(i);
        u32 pos = 0;
        for (u32 k = 0; k < tot; ++k) {
            if (k == i) continue;
            pos += before(line_at(k), x) ? 1u : 0u;
        }
        if (!ovr) {
            o_first[dst + pos] = mv.g_first[x];
            o_nlev[dst + pos] = mv.g_nlev[x];
            o_local[dst + pos] = mv.g_local[x];
            for (u32 lev = 0; lev < ML; ++lev) o_conf[(size_t)(dst + pos) * ML + lev] = mv.g_conf[(size_t)x * ML + lev];
        } else if (pos == 0) {  // signals of the best computed line, lineage and 1.0s of the exact match (raxtax.rs:73-84)
            const u32 id = b.exact_ids[b.exact_off[q]];
            const u32 n = ix.ref_levels[id];
            o_first[dst] = id;
            o_nlev[dst] = (u8)n;
            o_local[dst] = mv.g_local[x];
            for (u32 lev = 0; lev < ML; ++lev) o_conf[(size_t)dst * ML + lev] = lev < n ? 1.0 : 0.0;
        }
    }
}

// =========================================================================================================
// K5 (level-synchronous form, the default for unsharded indexes).  The depth-first walker above follows one chain of
// dependent loads per 32 children it looks at; taxonomies have nodes with thousands of children, so even a query with a
// single result line evaluates ~2 500 children (80 dependent round trips), and a query with a flat probability profile
// (40 orders above the cutoff, a 0.01 fallback chain under each) 78 000 of them -- that one walk set the kernel time
// (3.3 M cycles against a median of 0.11 M on C2).  Here a CTA of four warps owns a query and works level by level:
//   * the significant nodes of all levels are appended to a log in shared memory; the log range of one level is the
//     frontier, the children of the whole frontier are flattened (prefix sum of child counts + binary search) and every
//     warp evaluates 2 x 32 of them per step with independent loads;
//   * frontier entries without a significant child become a result (Taxon) or the head of a fallback chain (Inner,
//     lineage.rs:151-177); all chains advance together, one level per round, with a segmented arg-max over the
//     flattened children (last maximal child wins, ties as in the walker above);
//   * results are ordered by (confidence vector descending, first reference ascending): depth-first push order IS
//     ascending first reference, because emitted nodes own disjoint reference ranges and siblings ascend.  The order of
//     the log itself (shared-memory atomics) therefore does not matter.
// A query whose log or frontier would overflow is marked kQWalkRetry and redone by lineage_walk_kernel<false>.
// =========================================================================================================
constexpr u32 kBfsEntries = 512;   // significant nodes + fallback chain nodes of one query
constexpr u32 kBfsFrontier = 256;  // nodes of one level / simultaneously active fallback chains
// Large frontiers.  Taxonomies have giant nodes (a genus with 75 k species, an order with thousands of families), and enumerating the
// children of every frontier node made a flat-profile query test 250 k children per walk and even a one-line query 30-86 k.
//   * Significant children (lineage.rs:126-149) are found by a mass-pruned search instead: a run of children whose total probability
//     mass stays below 0.005 cannot contain a child with round(conf * 100) != 0, so a warp cuts a run into 32 sub-runs, reads the 33
//     prefix values at their ends and keeps the sub-runs that reach the floor; runs of at most kBfsLeaf children ("pairs": node +
//     child run) are then evaluated child by child exactly as before.  Disjoint runs of mass >= 0.005: at most 200 per round.
//   * The fallback arg-max (lineage.rs:156-164) has no such bound -- every child of a chain head has to be looked at -- except for a
//     query that kept few 512-reference segments (K4's mass cut): children wholly inside dropped segments are exactly 0, and the
//     runs that overlap a kept segment are found by binary search over the head's sorted child ranges (bfs_build_pairs).
constexpr u32 kBfsKept = 128;                         // more kept segments than this: the arg-max looks at every child (flat profiles)
constexpr u32 kBfsPairs = 512;                        // >= kBfsFrontier + max(kBfsKept, 200)
constexpr u32 kBfsPairMin = 768;                      // frontiers with fewer children are enumerated as before
constexpr u32 kBfsSmallNode = 48;                     // arg-max pairs: a node with so few children is one pair, no search
constexpr u32 kBfsLeaf = 64;                          // search: runs this short are evaluated child by child
constexpr u32 kBfsQueue = 256;                        // search: runs in flight per round
constexpr double kBfsMassFloor = 0.004999;            // a child is significant from 0.005 on; the margin covers the rounding of the sums
constexpr int kBfsThreads = 256;  // CTA size of lineage_bfs_kernel
constexpr int kBfsWarps = kBfsThreads / 32;
constexpr u32 kBfsPtabSmemMax = 16384;   // the query's P(m) table is staged behind BfsSmem when it fits (K <= 2047), see bfs_ptab_smem
__host__ __device__ inline size_t bfs_ptab_smem(u32 hstride) { return (size_t)hstride * 8 <= kBfsPtabSmemMax ? (size_t)hstride * 8 : 0; }
// ... and so is its skip bitmap (one bit per 512-reference segment)
__host__ __device__ inline size_t bfs_skip_smem(u64 n_pad) { return (size_t)(((n_pad / 512 + 31) / 32 * 4 + 15) & ~(u64)15); }

struct BfsSmem {
    unsigned long long* best;  // [F] arg-max value (bits of a non-negative double)
    double* res_local;         // [R]
    u32* ent_cf;               // [E]
    u32* ent_cc;               // [E] child_count | type << 30
    u32* ent_lo;               // [E]
    u32* ent_size;             // [E]
    u32* fr_off;               // [P + 1] offsets of the flattened children, per frontier node or per pair
    u32* besti;                // [F]
    u32* pair_a;               // [P] first child of the pair's run
    u32* pair_b;               // [P] one past its last child
    u32* pbase;                // [F + 1] first pair of a frontier node
    u32* kept;                 // [kBfsKept] kept segments, ascending
    u32* q_a;                  // [2][kBfsQueue] search runs (current / next round): first child,
    u32* q_b;                  // [2][kBfsQueue] one past the last child,
    u16* ent_parent;           // [E]
    u16* list_a;               // [F] fallback heads / active chains (current)
    u16* list_b;               // [F] active chains (next)
    u16* res_ent;              // [R]
    u16* order;                // [R]
    u16* pair_own;             // [P] frontier position of the pair's node
    u16* pj0;                  // [F] first kept segment under a frontier node
    u16* q_own;                // [2][kBfsQueue] frontier position of the run's node
    u16* ent_sj;               // [E] sharded walk: 1 + straddler index of the node, 0 = it lies inside this shard
    u8* ent_k;                 // [E]
    u8* ent_depth;             // [E]
    u8* ent_any;               // [E]
    u8* res_k;                 // [R][ML]
    static constexpr u32 E = kBfsEntries, F = kBfsFrontier, R = RTX_MAX_RESULTS_PER_QUERY, P = kBfsPairs;
    __host__ __device__ static size_t bytes(u32 ML) {
        size_t b = (size_t)F * 8 + (size_t)R * 8 + (size_t)E * 16 + (size_t)(P + 1) * 4 + (size_t)F * 4 + (size_t)P * 8 + (size_t)(F + 1) * 4 +
                   (size_t)kBfsKept * 4 + (size_t)kBfsQueue * 20 + (size_t)E * 4 + (size_t)F * 4 + (size_t)R * 4 + (size_t)P * 2 + (size_t)F * 2 + (size_t)E * 3 +
                   (size_t)R * ML;
        return (b + 64 + 15) & ~(size_t)15;
    }
    __device__ BfsSmem(unsigned char* base, u32 ML) {
        best = reinterpret_cast<unsigned long long*>(base);
        res_local = reinterpret_cast<double*>(best + F);
        ent_cf = reinterpret_cast<u32*>(res_local + R);
        ent_cc = ent_cf + E;
        ent_lo = ent_cc + E;
        ent_size = ent_lo + E;
        fr_off = ent_size + E;
        besti = fr_off + P + 1;
        pair_a = besti + F;
        pair_b = pair_a + P;
        pbase = pair_b + P;
        kept = pbase + F + 1;
        q_a = kept + kBfsKept;
        q_b = q_a + 2 * kBfsQueue;
        ent_parent = reinterpret_cast<u16*>(q_b + 2 * kBfsQueue);
        list_a = ent_parent + E;
        list_b = list_a + F;
        res_ent = list_b + F;
        order = res_ent + R;
        pair_own = order + R;
        pj0 = pair_own + P;
        q_own = pj0 + F;
        ent_sj = q_own + 2 * kBfsQueue;
        ent_k = reinterpret_cast<u8*>(ent_sj + E);
        ent_depth = ent_k + E;
        ent_any = ent_depth + E;
        res_k = ent_any + E;
    }
};

// warp 0: exclusive prefix of the child counts of `n` log entries (given by index list or by a contiguous range) -> fr_off[0..n]
// (skip_strad: entries of straddling nodes count no children -- fallback rounds of the sharded walk)
__device__ __forceinline__ void bfs_child_offsets(const BfsSmem& w, u32 n, u32 range_begin, const u16* __restrict__ list, int lane,
                                                  bool skip_strad = false) {
    u32 running = 0;
    for (u32 bb = 0; bb < n; bb += 32) {
        const u32 i = bb + lane;
        const u32 e = (i < n) ? (list ? (u32)list[i] : range_begin + i) : 0u;
        const u32 c = (i < n && !(skip_strad && w.ent_sj[e])) ? (w.ent_cc[e] & 0x3FFFFFFFu) : 0u;
        const u32 inc = warp_scan_incl(c, lane);
        if (i < n) w.fr_off[i] = running + inc - c;
        running += __shfl_sync(kFullMask, inc, 31);
    }
    if (lane == 0) w.fr_off[n] = running;
}
// largest i in [0, n) with fr_off[i] <= idx (entries without children share their successor's offset and are skipped)
__device__ __forceinline__ u32 bfs_owner(const u32* __restrict__ fr_off, u32 n, u32 idx) {
    u32 lo = 0, hi = n;
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (fr_off[mid] <= idx) lo = mid;
        else hi = mid;
    }
    return lo;
}

// first index in the ascending list `a[0..n)` whose value is >= key
__device__ __forceinline__ u32 bfs_lower_bound(const u32* __restrict__ a, u32 n, u32 key) {
    u32 lo = 0, hi = n;
    while (lo < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// Sparse expansion of `n` frontier nodes (log entries given by index list or by a contiguous range): the pairs (node, kept segment
// under it) with the run of the node's children that overlaps the segment -> pair_own / pair_a, fr_off[0..P] = offsets of the runs in
// the flattened child list.  Runs of one node are clipped against their predecessor, so no child appears twice.  Children are sorted
// and disjoint (tree.rs:77-107), their [lo, lo + size) are read from the node records.  Block-wide (four barriers); returns P.
// (shard_begin: first reference of this shard -- segments count local references; skip_strad as in bfs_child_offsets)
__device__ u32 bfs_build_pairs(const BfsSmem& w, const NodeRec* __restrict__ recs, u32 n, u32 range_begin, const u16* __restrict__ list,
                               u32 n_kept, int tid, u32 shard_begin, bool skip_strad, u32 small_node) {
    const int lane = tid & 31, warp = tid >> 5;
    for (u32 i = tid; i < n; i += kBfsThreads) {
        const u32 e = list ? (u32)list[i] : range_begin + i;
        const u32 cc = (skip_strad && w.ent_sj[e]) ? 0u : (w.ent_cc[e] & 0x3FFFFFFFu);
        const u32 lo = w.ent_lo[e] - shard_begin, hi = lo + w.ent_size[e];  // (nodes inside the shard)
        const u32 j0 = bfs_lower_bound(w.kept, n_kept, lo / kPrefixSeg);
        const u32 j1 = bfs_lower_bound(w.kept, n_kept, (hi + kPrefixSeg - 1) / kPrefixSeg);
        u32 np = (cc == 0 || j1 <= j0) ? 0u : j1 - j0;
        if (cc <= small_node) np = min(np, 1u);
        w.pj0[i] = (u16)j0;
        w.besti[i] = np;  // (the fallback rounds initialise besti behind this call)
    }
    __syncthreads();
    if (warp == 0) {
        u32 running = 0;
        for (u32 bb = 0; bb < n; bb += 32) {
            const u32 i = bb + lane;
            const u32 c = (i < n) ? w.besti[i] : 0u;
            const u32 inc = warp_scan_incl(c, lane);
            if (i < n) w.pbase[i] = running + inc - c;
            running += __shfl_sync(kFullMask, inc, 31);
        }
        if (lane == 0) w.pbase[n] = running;
    }
    __syncthreads();
    const u32 P = w.pbase[n];
    for (u32 t = tid; t < 2 * P; t += kBfsThreads) {
        const u32 p = t >> 1, upper = t & 1u;
        const u32 i = bfs_owner(w.pbase, n, p);
        const u32 e = list ? (u32)list[i] : range_begin + i;
        const u32 cf = w.ent_cf[e], cc = w.ent_cc[e] & 0x3FFFFFFFu;
        u32 val;
        if (cc <= small_node) {
            val = upper ? cc : 0u;
        } else {
            const u32 seg = w.kept[(u32)w.pj0[i] + (p - w.pbase[i])];
            // lower: first child that ends behind the segment's first reference; upper: first child that starts behind its last one
            const u64 key = (u64)shard_begin + (upper ? ((u64)seg + 1u) * kPrefixSeg : (u64)seg * kPrefixSeg);
            u32 lo = 0, hi = cc;
            while (lo < hi) {
                const u32 mid = (lo + hi) >> 1;
                const uint2 ls = *reinterpret_cast<const uint2*>(&recs[cf + mid].lo);  // lo, size
                const bool right = upper ? ((u64)ls.x >= key) : ((u64)ls.x + ls.y > key);
                if (right) hi = mid;
                else lo = mid + 1;
            }
            val = lo;
        }
        if (upper) {
            w.pair_b[p] = val;
        } else {
            w.pair_a[p] = val;
            w.pair_own[p] = (u16)i;
        }
    }
    __syncthreads();
    if (warp == 0) {
        u32 running = 0;
        for (u32 bb = 0; bb < P; bb += 32) {
            const u32 p = bb + lane;
            u32 a = 0, c = 0;
            if (p < P) {
                a = w.pair_a[p];
                if (p > 0 && w.pair_own[p - 1] == w.pair_own[p]) a = max(a, w.pair_b[p - 1]);  // pair_b ascends within a node
                const u32 bx = w.pair_b[p];
                c = bx > a ? bx - a : 0u;
            }
            const u32 inc = warp_scan_incl(c, lane);
            __syncwarp();
            if (p < P) {
                w.pair_a[p] = a;
                w.fr_off[p] = running + inc - c;
            }
            running += __shfl_sync(kFullMask, inc, 31);
        }
        if (lane == 0) w.fr_off[P] = running;
    }
    __syncthreads();
    return P;
}

// probability mass in front of child j of a node (j == cc: behind its last child), see node_conf
__device__ __forceinline__ double bfs_child_prefix(const NodeRec* __restrict__ recs, u32 cf, u32 cc, u32 j, const MassView& mv) {
    const bool end = j >= cc;
    const NodeRec* r = recs + cf + (end ? cc - 1u : j);
    const uint2 bb = *reinterpret_cast<const uint2*>(&r->blo), ss = *reinterpret_cast<const uint2*>(&r->slo);
    const u32 p = end ? bb.y : bb.x, si = end ? ss.y : ss.x;
    return mv.segoff[si] + mass_rel(mv, p, si);
}

// Mass-pruned search for the child runs of `n` frontier nodes (log entries range_begin ..) that can hold a significant child ->
// pair_own / pair_a, fr_off[0..P].  ctr: four shared counters (pairs, runs of this round, runs of the next, overflow).  Block-wide;
// returns P, or ~0u when a list overflowed (the caller hands the query to the depth-first walker).
// SH (reference-sharded walk): the prefixes only know this shard's references.  Of a large node's children those that touch the shard
// [sh_lo, sh_hi) are found by binary search; the first and the last of them may straddle a cut (their confidence comes from the
// combined records) and are always looked at, the ones in between lie inside the shard and are searched by mass.
template <bool SH>
__device__ u32 bfs_search_pairs(const BfsSmem& w, const NodeRec* __restrict__ recs, const MassView& mv, u32 n, u32 range_begin, u32* ctr, int tid,
                                u64 sh_lo, u64 sh_hi, u32 leaf_len) {
    const int lane = tid & 31, warp = tid >> 5;
    const u32 lt_mask = (1u << lane) - 1u;
    if (tid < 4) ctr[tid] = 0u;
    __syncthreads();
    for (u32 bb = 0; bb < n; bb += kBfsThreads) {  // small nodes are one pair each, the others start as one run
        const u32 i = bb + tid;
        const u32 cc = (i < n) ? (w.ent_cc[range_begin + i] & 0x3FFFFFFFu) : 0u;
        u32 np = 0, nq = 0, pa[2] = {0u, 0u}, pb[2] = {0u, 0u}, qa = 0, qb = 0;
        if (cc != 0 && cc <= leaf_len) {
            np = 1;
            pb[0] = cc;
        } else if (cc != 0) {
            u32 ta = 0, tb = cc;
            if (SH) {
                const u32 cf = w.ent_cf[range_begin + i];
                u32 lo = 0, hi = cc;
                while (lo < hi) {  // first child that ends behind the shard's first reference
                    const u32 mid = (lo + hi) >> 1;
                    const uint2 ls = *reinterpret_cast<const uint2*>(&recs[cf + mid].lo);
                    if ((u64)ls.x + ls.y > sh_lo) hi = mid;
                    else lo = mid + 1;
                }
                ta = lo;
                hi = cc;
                while (lo < hi) {  // first child that starts behind its last one
                    const u32 mid = (lo + hi) >> 1;
                    const uint2 ls = *reinterpret_cast<const uint2*>(&recs[cf + mid].lo);
                    if ((u64)ls.x >= sh_hi) hi = mid;
                    else lo = mid + 1;
                }
                tb = lo;
            }
            if (tb > ta && (tb - ta <= leaf_len)) {
                np = 1;
                pa[0] = ta;
                pb[0] = tb;
            } else if (tb > ta) {
                if (SH) {
                    np = 2;
                    pa[0] = ta;
                    pb[0] = ta + 1;
                    pa[1] = tb - 1;
                    pb[1] = tb;
                    ++ta;
                    --tb;
                }
                nq = 1;
                qa = ta;
                qb = tb;
            }
        }
        const u32 pinc = warp_scan_incl(np, lane);
        const u32 ptot = __shfl_sync(kFullMask, pinc, 31);
        const u32 mb = __ballot_sync(kFullMask, nq != 0);
        u32 ps = 0, pq = 0;
        if (lane == 0) {
            if (ptot) ps = atomicAdd(&ctr[0], ptot);
            if (mb) pq = atomicAdd(&ctr[1], (u32)__popc(mb));
        }
        ps = __shfl_sync(kFullMask, ps, 0);
        pq = __shfl_sync(kFullMask, pq, 0);
        if (ps + ptot > kBfsPairs || pq + __popc(mb) > kBfsQueue) {
            if (lane == 0) ctr[3] = 1u;
        } else {
            const u32 pos = ps + pinc - np;
            for (u32 k = 0; k < np; ++k) {
                w.pair_own[pos + k] = (u16)i;
                w.pair_a[pos + k] = pa[k];
                w.pair_b[pos + k] = pb[k];
            }
            if (nq) {
                const u32 qp = pq + __popc(mb & lt_mask);
                w.q_own[qp] = (u16)i;
                w.q_a[qp] = qa;
                w.q_b[qp] = qb;
            }
        }
    }
    __syncthreads();
    u32 cur = 0;
    while (true) {  // block-uniform
        const u32 n_in = ctr[1 + cur];
        if (n_in == 0 || ctr[3]) break;
        const u32 nxt = cur ^ 1u;
        for (u32 it = warp; it < n_in; it += kBfsWarps) {
            const u32 own = w.q_own[cur * kBfsQueue + it], a = w.q_a[cur * kBfsQueue + it], b = w.q_b[cur * kBfsQueue + it];
            const u32 e = range_begin + own;
            const u32 cf = w.ent_cf[e], cc = w.ent_cc[e] & 0x3FFFFFFFu;
            const u32 step = (b - a + 31u) / 32u;
            const u32 sa = min(a + (u32)lane * step, b), sb = min(sa + step, b);
            const double v0 = bfs_child_prefix(recs, cf, cc, sa, mv);
            double v1 = __shfl_down_sync(kFullMask, v0, 1);
            if (lane == 31) v1 = bfs_child_prefix(recs, cf, cc, sb, mv);
            const bool keep = sa < sb && (v1 - v0) >= kBfsMassFloor;
            const bool leaf = keep && sb - sa <= leaf_len, more = keep && !leaf;
            const u32 ml = __ballot_sync(kFullMask, leaf), mm = __ballot_sync(kFullMask, more);
            u32 pl = 0, pm = 0;
            if (lane == 0) {
                if (ml) pl = atomicAdd(&ctr[0], (u32)__popc(ml));
                if (mm) pm = atomicAdd(&ctr[1 + nxt], (u32)__popc(mm));
            }
            pl = __shfl_sync(kFullMask, pl, 0);
            pm = __shfl_sync(kFullMask, pm, 0);
            if (pl + __popc(ml) > kBfsPairs || pm + __popc(mm) > kBfsQueue) {
                if (lane == 0) ctr[3] = 1u;
            } else if (leaf) {
                const u32 pos = pl + __popc(ml & lt_mask);
                w.pair_own[pos] = (u16)own;
                w.pair_a[pos] = sa;
                w.pair_b[pos] = sb;
            } else if (more) {
                const u32 pos = nxt * kBfsQueue + pm + __popc(mm & lt_mask);
                w.q_own[pos] = (u16)own;
                w.q_a[pos] = sa;
                w.q_b[pos] = sb;
            }
        }
        __syncthreads();
        if (tid == 0) ctr[1 + cur] = 0u;
        cur = nxt;
        __syncthreads();
    }
    if (ctr[3]) return ~0u;
    const u32 P = ctr[0];
    if (warp == 0) {
        u32 running = 0;
        for (u32 bb = 0; bb < P; bb += 32) {
            const u32 p = bb + lane;
            const u32 c = (p < P) ? w.pair_b[p] - w.pair_a[p] : 0u;
            const u32 inc = warp_scan_incl(c, lane);
            if (p < P) w.fr_off[p] = running + inc - c;
            running += __shfl_sync(kFullMask, inc, 31);
        }
        if (lane == 0) w.fr_off[P] = running;
    }
    __syncthreads();
    return P;
}

// SH: the reference-sharded walk (see lineage_walk_kernel<true> for the rules): a child that straddles a shard cut takes its confidence
// from the combined records, a child inside another shard is left to its owner; a straddling node learns from the combined flags whether
// it has a significant child / whether a line is pushed below it, and is reported by the rank that holds its first reference; a fallback
// chain follows the combined best child through straddling nodes and ends where it leaves the shard.
template <bool SH>
__global__ void __launch_bounds__(kBfsThreads)  // (a 6-CTA/SM bound, 40 registers with small spills, measured the same 0.89 ms)
    lineage_bfs_kernel(IndexView ix, const NodeRec* __restrict__ recs, BatchView b, ResultPool pool, ProbScratch sc, ShardView sv, int q_base,
                       int q_count, u32 entry_cap, int sparse) {
    extern __shared__ __align__(16) unsigned char bsm_raw[];
    __shared__ u32 s_log_n, s_n_res, s_n_fb, s_n_next, s_retry, s_retry_cls;  // s_retry_cls: raised while sorting a frontier (see the level loop)
    __shared__ u32 s_n_kept;  // kept segments of a sparse query, 0 = the arg-max looks at every child
    __shared__ u32 s_ctr[4], s_slow;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ql = blockIdx.x;
    if (ql >= q_count) return;
    const int q = q_base + ql;
    const u32 ML = ix.max_levels;
    BfsSmem w(bsm_raw, ML);
    constexpr u32 F = BfsSmem::F, R = BfsSmem::R;
    const u32 E = min(BfsSmem::E, entry_cap);  // a smaller cap only serves the tests of the retry path
    const double Nd = (double)ix.n_refs;
    MassView mv = mass_view(sc, ql);
    if (bfs_ptab_smem(b.hstride)) {  // the gathers of node_conf / mass_rel then come from shared memory (visible behind the first barrier below)
        double* ptab_s = reinterpret_cast<double*>(bsm_raw + BfsSmem::bytes(ML));
        const u32 K1 = (u32)b.K[q] + 1u;
        for (u32 m = tid; m < K1; m += kBfsThreads) ptab_s[m] = mv.ptab[m];
        mv.ptab = ptab_s;
    }
    {
        u32* skip_s = reinterpret_cast<u32*>(bsm_raw + BfsSmem::bytes(ML) + bfs_ptab_smem(b.hstride));
        const u32 n_words = (u32)((ix.n_pad / kPrefixSeg + 31) / 32);
        for (u32 i = tid; i < n_words; i += kBfsThreads) skip_s[i] = mv.skipw[i];
        mv.skipw = skip_s;
    }
    __syncthreads();  // (block-uniform: the tables are read by warp 0 right below)
    const u32 lt_mask = (1u << lane) - 1u;
    const u64 sh_lo = ix.shard_begin, sh_hi = ix.shard_begin + ix.shard_refs;
    auto inside = [&](const NodeRec& r) { return (u64)r.lo >= sh_lo && (u64)r.lo + r.size <= sh_hi; };
    auto owned = [&](u32 lo) { return (u64)lo >= sh_lo && (u64)lo < sh_hi; };  // this rank reports a straddling node that starts here
    const size_t srow = SH ? (size_t)ql * sv.n_strad : 0;
    // sparse == 2 (test hook): the large-frontier paths run on every frontier, with runs of two children
    const u32 pair_min = sparse == 2 ? 0u : kBfsPairMin, leaf_len = sparse == 2 ? 2u : kBfsLeaf, small_node = sparse == 2 ? 2u : kBfsSmallNode;
    int status = pool.status[q];

    u32 n_res = 0;
    if (status == kQOk) {  // block-uniform
        if (tid == 0) {
            const NodeRec root = recs[0];
            w.ent_sj[0] = SH ? (u16)(sv.strad_of_node[0] + 1) : (u16)0;
            w.ent_cf[0] = root.child_first;
            w.ent_cc[0] = root.cc_type;
            w.ent_lo[0] = root.lo;
            w.ent_size[0] = root.size;
            w.ent_parent[0] = 0xFFFFu;
            w.ent_k[0] = 0;
            w.ent_depth[0] = 0;
            w.ent_any[0] = 0;
            s_log_n = 1;
            s_n_res = 0;
            s_n_fb = 0;
            s_retry = 0;
            s_retry_cls = 0;
        }
        if (warp == 0) {  // the kept segments (K4's skip bitmap, complemented), in ascending order, if they are few
            const u32 n_seg = (u32)(ix.n_pad / kPrefixSeg), n_words = (n_seg + 31u) / 32u;
            u32 running = 0;
            bool few = sparse != 0;
            for (u32 bb = 0; bb < n_words && few; bb += 32) {
                const u32 wi = bb + lane;
                u32 kw = 0;
                if (wi < n_words) {
                    kw = ~mv.skipw[wi];
                    if (wi * 32u + 32u > n_seg) kw &= (1u << (n_seg - wi * 32u)) - 1u;  // (n_seg is not a multiple of 32 here)
                }
                const u32 c = __popc(kw);
                const u32 inc = warp_scan_incl(c, lane);
                const u32 tot = __shfl_sync(kFullMask, inc, 31);
                if (running + tot > kBfsKept) {
                    few = false;
                } else {
                    u32 pos = running + inc - c;
                    while (kw) {
                        w.kept[pos++] = wi * 32u + (u32)__ffs(kw) - 1u;
                        kw &= kw - 1u;
                    }
                    running += tot;
                }
            }
            if (lane == 0) s_n_kept = few ? running : 0u;
        }
        __syncthreads();
        const u32 n_kept = s_n_kept;
        // ---- significant nodes, level by level (lineage.rs:126-149).  Two barriers per level: the child offsets of the current
        // frontier (warp 0) are computed in the same phase in which the previous frontier is sorted into result lines and
        // fallback heads (its ent_any flags are final since the barrier behind the evaluation that set them).  Each phase has its
        // own overflow flag -- s_retry_cls is written before the first barrier and read behind it, s_retry between the barriers and
        // read behind the second -- so that no warp can test a flag another warp is raising in the same phase -------------
        u32 lvl_begin = 0, lvl_end = 1, prev_begin = 0, prev_end = 0;
#ifdef RTX_WALK_TRACE
        const long long tr_t0 = clock64();
        long long tr_lvl_t[12];
        u32 tr_lvl_tot[12], tr_lvl_nf[12], tr_nl = 0, tr_fb_children = 0, tr_fb_rounds = 0, tr_fb_heads = 0;
#endif
        while (true) {
#ifdef RTX_WALK_TRACE
            const long long tr_a = clock64();
#endif
            const bool have = lvl_begin < lvl_end;
            const u32 nf = lvl_end - lvl_begin;
            if (have && warp == 0) bfs_child_offsets(w, nf, lvl_begin, nullptr, lane);
            // entries of the previous frontier without a significant child: Taxon -> result line, Inner -> head of a fallback chain
            const u32 pn = prev_end - prev_begin;
            for (u32 bb = 0; bb < pn; bb += kBfsThreads) {
                const u32 i = bb + tid;
                bool is_res = false, is_fb = false;
                const u32 e = prev_begin + i;
                if (i < pn) {
                    bool any_sig = w.ent_any[e] != 0, pushed = any_sig, mine = true;
                    if (SH && w.ent_sj[e]) {
                        const u32 sa = sv.sany[srow + w.ent_sj[e] - 1u];
                        any_sig = any_sig || (sa & 1u);
                        pushed = pushed || (sa & 2u);
                        mine = owned(w.ent_lo[e]);
                    }
                    const u32 type = w.ent_cc[e] >> 30;
                    is_fb = type == 0 && !any_sig;
                    is_res = type == 1 && e != 0 && !pushed && mine;  // the root never reports itself
                }
                const u32 mr = __ballot_sync(kFullMask, is_res), mf = __ballot_sync(kFullMask, is_fb);
                u32 pr = 0, pf = 0;
                if (lane == 0) {
                    if (mr) pr = atomicAdd(&s_n_res, (u32)__popc(mr));
                    if (mf) pf = atomicAdd(&s_n_fb, (u32)__popc(mf));
                }
                pr = __shfl_sync(kFullMask, pr, 0);
                pf = __shfl_sync(kFullMask, pf, 0);
                if (pr + __popc(mr) > R || pf + __popc(mf) > F) {
                    if (lane == 0) s_retry_cls = 1;
                } else {
                    if (is_res) w.res_ent[pr + __popc(mr & lt_mask)] = (u16)e;
                    if (is_fb) w.list_a[pf + __popc(mf & lt_mask)] = (u16)e;
                }
            }
            __syncthreads();
            if (!have || s_retry_cls) break;
            u32 total = w.fr_off[nf], n_own = nf;
            const bool pairs = sparse != 0 && total >= pair_min;  // block-uniform
            if (pairs) {
                n_own = bfs_search_pairs<SH>(w, recs, mv, nf, lvl_begin, s_ctr, tid, sh_lo, sh_hi, leaf_len);
                if (n_own == ~0u) {  // (every thread sees the same return value)
                    if (tid == 0) s_retry = 1;
                    break;
                }
                total = w.fr_off[n_own];
            }
            for (u32 base = (u32)warp * 64; base < total; base += kBfsWarps * 64) {  // two chunks of 32 children in flight per warp
                u32 kk[2], ee[2];
                int sj[2];
                NodeRec cr[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const u32 idx = base + u * 32 + lane;
                    ee[u] = 0;
                    sj[u] = -1;
                    cr[u] = NodeRec{0, 0, 0, 0, 0, 0, 0, 0};
                    if (idx < total) {
                        const u32 o = bfs_owner(w.fr_off, n_own, idx);
                        ee[u] = lvl_begin + (pairs ? (u32)w.pair_own[o] : o);
                        const u32 cn = w.ent_cf[ee[u]] + (pairs ? w.pair_a[o] : 0u) + (idx - w.fr_off[o]);
                        cr[u] = recs[cn];
                        if (SH) sj[u] = sv.strad_of_node[cn];
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const u32 idx = base + u * 32 + lane;
                    kk[u] = 0u;
                    if (idx < total) {
                        if (SH && sj[u] >= 0) kk[u] = sv.sk[srow + sj[u]];  // combined over the ranks
                        else if (!SH || inside(cr[u])) kk[u] = (u32)round(node_conf(mv, cr[u]) * 100.0);  // f64::round (lineage.rs:129)
                        // children inside another shard are walked by their owner
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const u32 mask = __ballot_sync(kFullMask, kk[u] != 0);
                    if (mask) {
                        u32 pos0 = 0;
                        if (lane == 0) pos0 = atomicAdd(&s_log_n, (u32)__popc(mask));
                        pos0 = __shfl_sync(kFullMask, pos0, 0);
                        if (pos0 + __popc(mask) > E) {
                            if (lane == 0) s_retry = 1;
                        } else if (kk[u] != 0) {
                            const u32 pos = pos0 + __popc(mask & lt_mask);
                            w.ent_cf[pos] = cr[u].child_first;
                            w.ent_cc[pos] = cr[u].cc_type;
                            w.ent_lo[pos] = cr[u].lo;
                            w.ent_size[pos] = cr[u].size;
                            w.ent_parent[pos] = (u16)ee[u];
                            w.ent_k[pos] = (u8)min(kk[u], 255u);
                            w.ent_depth[pos] = (u8)(w.ent_depth[ee[u]] + 1);
                            w.ent_any[pos] = 0;
                            w.ent_any[ee[u]] = 1;
                            w.ent_sj[pos] = (u16)(sj[u] + 1);
                            // a significant Sequence node (it has children, or it would not be in the tree) may push nothing, and
                            // its Taxon parent is then reported after all (lineage.rs:143-149): the depth-first walker tracks that
                            if ((cr[u].cc_type >> 30) == 2u) s_retry = 1;
                        }
                    }
                }
            }
            __syncthreads();
#ifdef RTX_WALK_TRACE
            if (tr_nl < 12) {
                tr_lvl_t[tr_nl] = clock64() - tr_a;
                tr_lvl_tot[tr_nl] = total;
                tr_lvl_nf[tr_nl] = nf | (pairs ? 0x80000000u : 0u);
                ++tr_nl;
            }
#endif
            if (s_retry) break;
            prev_begin = lvl_begin;
            prev_end = lvl_end;
            lvl_begin = lvl_end;
            lvl_end = s_log_n;  // stable: nothing appends to the log before the next evaluation phase
            if (lvl_end - lvl_begin > F) {  // block-uniform
                if (tid == 0) s_retry = 1;
                break;
            }
        }
        __syncthreads();
        if (tid == 0 && s_retry_cls) s_retry = 1;
        __syncthreads();
        // ---- fallback chains (lineage.rs:151-177): all heads advance together, one level per round -------------------
        u16* cur = w.list_a;
        u16* nxt = w.list_b;
        u32 n_ch = s_retry ? 0u : s_n_fb;
#ifdef RTX_WALK_TRACE
        const long long tr_t1 = clock64();
        tr_fb_heads = n_ch;
#endif
        while (n_ch > 0) {  // block-uniform
            if (warp == 0) bfs_child_offsets(w, n_ch, 0, cur, lane, SH);
            if (tid == 0) s_n_next = 0;
            __syncthreads();
            u32 total = w.fr_off[n_ch], n_own = n_ch;
            const bool pairs = n_kept != 0 && total >= pair_min;  // block-uniform
            if (pairs) {
                n_own = bfs_build_pairs(w, recs, n_ch, 0, cur, n_kept, tid, (u32)sh_lo, SH, small_node);
                total = w.fr_off[n_own];
            }
            for (u32 i = tid; i < n_ch; i += kBfsThreads) {
                w.best[i] = 0ull;
                w.besti[i] = 0u;  // 1 + child index of the chain's last "record" (below); bit 31: the chain takes the second pass
            }
            if (tid == 0) s_slow = 0;
#ifdef RTX_WALK_TRACE
            tr_fb_children += total;
            ++tr_fb_rounds;
#endif
            __syncthreads();
            // max_by(partial_cmp): the LAST maximal child wins (lineage.rs:156-164); children tied in exact arithmetic (same hit counts)
            // differ only by rounding noise of the prefix sums, so values within 1e-12 relative of the maximum count as maximal.
            // One pass: a child within the tolerance of the running maximum of its chain is a "record"; every child within the
            // tolerance of the FINAL maximum is one (the running maximum only grows), so the record with the largest index is the
            // answer if it passes the final test itself -- else (values in the 1e-12 band right below the tolerance: practically
            // never) the chain is scanned a second time.  A warp whose 32 children belong to one chain (the giant nodes that carry the
            // cost) reduces first and touches shared memory twice.
            for (u32 base = 0; base < total; base += 2 * kBfsThreads) {  // two children per lane in flight
                bool valid[2];
                u32 c[2], ci[2];
                NodeRec cr[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const u32 idx = base + u * kBfsThreads + tid;
                    valid[u] = idx < total;
                    c[u] = 0;
                    ci[u] = 0;
                    cr[u] = NodeRec{0, 0, 0, 0, 0, 0, 0, 0};
                    if (valid[u]) {
                        const u32 o = bfs_owner(w.fr_off, n_own, idx);
                        c[u] = pairs ? (u32)w.pair_own[o] : o;
                        ci[u] = (pairs ? w.pair_a[o] : 0u) + (idx - w.fr_off[o]);
                        cr[u] = recs[w.ent_cf[cur[c[u]]] + ci[u]];
                    }
                }
                double vv[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) vv[u] = valid[u] ? fmax(node_conf(mv, cr[u]), 0.0) : 0.0;
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const double v = vv[u];
                    const u32 vm = __ballot_sync(kFullMask, valid[u]);
                    if (vm == 0u) continue;  // warp-uniform
                    const u32 c0 = __shfl_sync(kFullMask, c[u], __ffs(vm) - 1);
                    if (__all_sync(kFullMask, !valid[u] || c[u] == c0)) {
                        double vmax = v;  // (invalid lanes hold 0.0, the smallest admissible value)
#pragma unroll
                        for (int o2 = 16; o2 > 0; o2 >>= 1) vmax = fmax(vmax, __shfl_xor_sync(kFullMask, vmax, o2));
                        unsigned long long old = 0ull;
                        if (lane == 0) old = atomicMax(&w.best[c0], (unsigned long long)__double_as_longlong(vmax));  // non-negative doubles order like their bits
                        old = __shfl_sync(kFullMask, old, 0);
                        const double run = fmax(__longlong_as_double((long long)old), vmax);
                        const bool rec = valid[u] && v >= run - fabs(run) * 1e-12;
                        const u32 r = __reduce_max_sync(kFullMask, rec ? ci[u] + 1u : 0u);
                        if (lane == 0 && r) atomicMax(&w.besti[c0], r);
                    } else if (valid[u]) {
                        const unsigned long long old = atomicMax(&w.best[c[u]], (unsigned long long)__double_as_longlong(v));
                        const double run = fmax(__longlong_as_double((long long)old), v);
                        if (v >= run - fabs(run) * 1e-12) atomicMax(&w.besti[c[u]], ci[u] + 1u);
                    }
                }
            }
            __syncthreads();
            for (u32 i = tid; i < n_ch; i += kBfsThreads) {  // does the last record pass the final test?
                const u32 head = cur[i];
                const u32 hcc = w.ent_cc[head] & 0x3FFFFFFFu;
                const double bestv = __longlong_as_double((long long)w.best[i]);
                if (SH && w.ent_sj[head]) {
                    // the best child of a straddling node was decided from all ranks' records
                    const u32 bn = sv.sbest[srow + w.ent_sj[head] - 1u];
                    w.besti[i] = bn >= w.ent_cf[head] ? bn - w.ent_cf[head] + 1u : 1u;
                } else if (w.best[i] == 0ull || w.besti[i] == 0u) {
                    // no child above 0: all of them tie and the last one wins (the children outside the kept segments, which the
                    // sparse expansion does not look at, are exactly 0 as well)
                    w.besti[i] = hcc;
                } else {
                    const NodeRec cr = recs[w.ent_cf[head] + w.besti[i] - 1u];
                    const double v = fmax(node_conf(mv, cr), 0.0);
                    if (!(v >= bestv - fabs(bestv) * 1e-12)) {
                        w.besti[i] = 0x80000000u;
                        s_slow = 1u;
                    }
                }
            }
            __syncthreads();
            if (s_slow) {  // block-uniform; second pass over the marked chains: the LAST child within 1e-12 relative of the maximum
                for (u32 idx = tid; idx < total; idx += kBfsThreads) {
                    const u32 o = bfs_owner(w.fr_off, n_own, idx);
                    const u32 c = pairs ? (u32)w.pair_own[o] : o;
                    if (!(w.besti[c] & 0x80000000u)) continue;
                    const u32 ci = (pairs ? w.pair_a[o] : 0u) + (idx - w.fr_off[o]);
                    const NodeRec cr = recs[w.ent_cf[cur[c]] + ci];
                    const double v = fmax(node_conf(mv, cr), 0.0);
                    const double bestv = __longlong_as_double((long long)w.best[c]);
                    if (v >= bestv - fabs(bestv) * 1e-12) atomicMax(&w.besti[c], 0x80000000u | (ci + 1u));
                }
                __syncthreads();
            }
            for (u32 bb = 0; bb < n_ch; bb += kBfsThreads) {  // one new log entry (0.01) per chain; Inner nodes stay active
                const u32 i = bb + tid;
                NodeRec br = NodeRec{0, 0, 0, 0, 0, 0, 0, 0};
                u32 head = 0;
                int bsj = -1;
                bool here = true, mine = true;  // sharded: does the chain go on / end on this rank?
                if (i < n_ch) {
                    head = cur[i];
                    const u32 b1 = w.besti[i] & 0x7FFFFFFFu;  // 1 + index of the chosen child
                    w.besti[i] = b1 ? b1 - 1u : 0u;
                    const u32 bn = w.ent_cf[head] + w.besti[i];
                    br = recs[bn];
                    if (SH) {
                        bsj = sv.strad_of_node[bn];
                        here = bsj >= 0 || inside(br);  // else the chain continues in another rank's shard
                        mine = bsj >= 0 ? owned(br.lo) : here;
                    }
                }
                const bool is_inner = (br.cc_type >> 30) == 0;
                const bool go_on = i < n_ch && is_inner && here;
                const bool done = i < n_ch && !is_inner && mine;
                const bool valid = go_on || done;
                const u32 mv = __ballot_sync(kFullMask, valid), mg = __ballot_sync(kFullMask, go_on), md = __ballot_sync(kFullMask, done);
                u32 pv = 0, pg = 0, pd = 0;
                if (lane == 0) {
                    if (mv) pv = atomicAdd(&s_log_n, (u32)__popc(mv));
                    if (mg) pg = atomicAdd(&s_n_next, (u32)__popc(mg));
                    if (md) pd = atomicAdd(&s_n_res, (u32)__popc(md));
                }
                pv = __shfl_sync(kFullMask, pv, 0);
                pg = __shfl_sync(kFullMask, pg, 0);
                pd = __shfl_sync(kFullMask, pd, 0);
                if (pv + __popc(mv) > E || pd + __popc(md) > R) {
                    if (lane == 0) s_retry = 1;
                } else if (valid) {
                    const u32 pos = pv + __popc(mv & lt_mask);
                    w.ent_cf[pos] = br.child_first;
                    w.ent_cc[pos] = br.cc_type;
                    w.ent_lo[pos] = br.lo;
                    w.ent_size[pos] = br.size;
                    w.ent_parent[pos] = (u16)head;
                    w.ent_k[pos] = 1;  // 1.0 / rounding_factor
                    w.ent_depth[pos] = (u8)(w.ent_depth[head] + 1);
                    w.ent_any[pos] = 0;
                    w.ent_sj[pos] = (u16)(bsj + 1);
                    if (go_on) nxt[pg + __popc(mg & lt_mask)] = (u16)pos;
                    else w.res_ent[pd + __popc(md & lt_mask)] = (u16)pos;
                }
            }
            __syncthreads();
            u16* t = cur;
            cur = nxt;
            nxt = t;
            n_ch = s_retry ? 0u : s_n_next;
            __syncthreads();
        }
        const bool retry = s_retry != 0;
#ifdef RTX_WALK_TRACE
        if (tid == 0) {
            const long long tr_t2 = clock64();
            if (tr_t2 - tr_t0 > 200000 || (q % 97) == 0) {
                printf("TR q %d kept %u retry %d res %u lvl_clk %lld fb_clk %lld heads %u rounds %u fbch %u |", q, n_kept, (int)retry, s_n_res, tr_t1 - tr_t0, tr_t2 - tr_t1,
                       tr_fb_heads, tr_fb_rounds, tr_fb_children);
                for (u32 i = 0; i < tr_nl; ++i) printf(" L%u nf %u%s ch %u clk %lld", i, tr_lvl_nf[i] & 0xFFFFu, (tr_lvl_nf[i] >> 31) ? "p" : "", tr_lvl_tot[i], tr_lvl_t[i]);
                printf("\n");
            }
        }
#endif
        n_res = retry ? 0u : s_n_res;
        // ---- confidence vectors and local signals of the result lines (lineage.rs:95-102, utils.rs:91-105) -------------
        bool too_deep = false;
        for (u32 r = warp; r < n_res; r += kBfsWarps) {
            const u32 e = w.res_ent[r];
            const int d = w.ent_depth[e];
            if (d > (int)ML || d > 32) {
                too_deep = true;
                continue;
            }
            double cv = 0.0, ev = 0.0;
            if (lane < d) {
                u32 c = e;
                for (int s2 = d - 1; s2 > lane; --s2) c = w.ent_parent[c];  // the path node of level `lane`
                cv = (double)w.ent_k[c] / 100.0;
                ev = (double)w.ent_size[c] / Nd;
                w.res_k[(size_t)r * ML + lane] = w.ent_k[c];
            }
            const u32 lt1 = __ballot_sync(kFullMask, lane < d && 1.0 > ev);
            const int start = lt1 ? (__ffs(lt1) - 1) : (d - 1);
            double a_sum = 0.0, b_sum = 0.0;  // sequential sums, level order, like the reference
            for (int i2 = start; i2 < d; ++i2) {
                a_sum += __shfl_sync(kFullMask, cv, i2);
                b_sum += __shfl_sync(kFullMask, ev, i2);
            }
            double s2 = 0.0;
            for (int i2 = start; i2 < d; ++i2) {
                const double df = __shfl_sync(kFullMask, cv, i2) / a_sum - __shfl_sync(kFullMask, ev, i2) / b_sum;
                s2 += df * df;
            }
            if (lane == 0) w.res_local[r] = sqrt(s2);
        }
        if (__syncthreads_or(too_deep ? 1 : 0) || retry) status = kQWalkRetry;
        else if (n_res == 0 && !SH) status = kQEmptyResult;  // assert!(!eval_res.is_empty()) raxtax.rs:72 (sharded: checked after the merge)
    }
    if (status == kQWalkRetry) {  // lineage_walk_kernel<false> redoes this query
        if (tid == 0) pool.status[q] = status;
        return;
    }
    // ---- order (lineage.rs:93): stable sort, descending lexicographic on the confidence vectors; the tie-break of the
    // reference's stable sort is the depth-first push order == ascending first reference
    if (status == kQOk) {
        for (u32 i = tid; i < n_res; i += kBfsThreads) {
            const u8* ci = w.res_k + (size_t)i * ML;
            const u32 li = w.ent_depth[w.res_ent[i]], fi = w.ent_lo[w.res_ent[i]];
            u32 rank = 0;
            for (u32 j = 0; j < n_res; ++j) {
                if (j == i) continue;
                const u8* cj = w.res_k + (size_t)j * ML;
                const u32 lj = w.ent_depth[w.res_ent[j]];
                int cmp = 0;  // +1: vector j > vector i
                for (u32 l = 0; l < min(li, lj); ++l) {
                    if (cj[l] != ci[l]) {
                        cmp = cj[l] > ci[l] ? 1 : -1;
                        break;
                    }
                }
                if (cmp == 0) cmp = (lj > li) ? 1 : (lj < li) ? -1 : 0;
                if (cmp > 0 || (cmp == 0 && w.ent_lo[w.res_ent[j]] < fi)) ++rank;
            }
            w.order[rank] = (u16)i;
        }
    }
    __syncthreads();
    // ---- override (raxtax.rs:73-84) and emission into the result pool ---------------------------------------
    u32 n_out = (status == kQOk) ? n_res : 0;
    bool ovr = false;
    u32 ovr_idx = 0;
    if (!SH && status == kQOk && !(b.flags & RTX_RAW_CONFIDENCE) && !(b.flags & RTX_SKIP_EXACT_MATCHES) && b.exact_off) {
        if (b.exact_off[q + 1] - b.exact_off[q] == 1) {  // sharded: the caller applies the override after merging the ranks
            ovr = true;
            ovr_idx = b.exact_ids[b.exact_off[q]];
            n_out = 1;
        }
    }
    __shared__ unsigned long long s_base;
    if (tid == 0) s_base = atomicAdd(pool.used, (unsigned long long)n_out);
    __syncthreads();
    const unsigned long long base = s_base;
    if (base + n_out > pool.cap) {
        if (status == kQOk) status = kQPoolOverflow;
    } else if (ovr) {
        const u32 nl = ix.ref_levels[ovr_idx];
        if (tid == 0) {
            pool.first_ref[base] = ovr_idx;
            pool.n_levels[base] = (u8)nl;
            pool.local[base] = w.res_local[w.order[0]];
        }
        for (u32 l = tid; l < ML; l += kBfsThreads) pool.conf[base * ML + l] = (l < nl) ? 1.0 : 0.0;
    } else {
        for (u32 x = tid; x < n_out * ML; x += kBfsThreads) {
            const u32 i = x / ML, l = x - i * ML;
            const u32 src = w.order[i];
            pool.conf[(base + i) * ML + l] = (l < w.ent_depth[w.res_ent[src]]) ? (double)w.res_k[(size_t)src * ML + l] / 100.0 : 0.0;
        }
        for (u32 i = tid; i < n_out; i += kBfsThreads) {
            const u32 src = w.order[i];
            pool.first_ref[base + i] = w.ent_lo[w.res_ent[src]];
            pool.n_levels[base + i] = w.ent_depth[w.res_ent[src]];
            pool.local[base + i] = w.res_local[src];
        }
    }
    if (tid == 0) {
        pool.res_off[q] = (u32)base;
        pool.res_cnt[q] = n_out;
        pool.status[q] = status;
    }
}

}  // namespace rtx
