// pss_kernels.cuh -- the sm_100a kernels of the pss-bam hot path.
//
//   pack_kernel      K6  ASCII contig -> 4-bit packed genome groups
//   spectrum_kernel / spectrum_smem16_kernel / radix_*_kernel
//                    K5  genome-kmer-count.c:68-79 + kmer.c:43-110 as a flat 4^k histogram
//   tally_kernel     K1-K4  SAM text tile -> records -> filters -> genome gather
//                           -> pss-bam count tables / fragkon end-context histograms
//
// Nothing here is GEMM shaped; the kernels are byte scans, gathers and
// histograms bound by HBM and by integer issue rate.  The per-record logic is
// in pss_record.h (shared with the CPU test build).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "pss_record.h"

namespace pssgpu {

// ---------------------------------------------------------------------------
// PTX: mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, size multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// one arrival at a counter in shared memory; returns the count before it.  Release: after a __syncwarp, the warp's
// earlier shared-memory accesses are ordered before the arrival; acquire: those of the earlier arrivals are ordered
// before what follows it.
__device__ __forceinline__ uint32_t arrive_count(uint32_t *ctr)
{
    uint32_t old;
    asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(ctr)) : "memory");
    return old;
}

// L2 prefetch of [src, src + bytes): size multiple of 16, address 16-byte aligned
__device__ __forceinline__ void bulk_prefetch_l2(const void *src_gmem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}

// ===========================================================================
// K6  genome pack
// ===========================================================================
struct PackArgs {
    const uint8_t *src;        // ASCII of bases [0, n_bases) of this piece (device)
    uint64_t       n_bases;
    uint64_t      *dst;        // first group of the piece
    uint64_t       gbase;      // global base index of src[0] (multiple of 16)
    uint64_t      *exc_pos;    // "other" symbol log
    uint8_t       *exc_chr;
    unsigned long long *exc_n;
    uint64_t       exc_cap;
    uint32_t      *flags;      // bit 0: NUL byte seen
};

__global__ void __launch_bounds__(256) pack_kernel(PackArgs A)
{
    const uint64_t n_groups = (A.n_bases + 15) / 16;
    const bool     aligned = ((uintptr_t)A.src & 15u) == 0;
    for (uint64_t gi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; gi < n_groups;
         gi += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t b0 = gi * 16;
        const int      nv = (A.n_bases - b0 >= 16) ? 16 : (int)(A.n_bases - b0);
        uint32_t       om = 0, nul = 0;
        uint64_t       grp;
        if (aligned && nv == 16) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(A.src + b0));
            const uint32_t w[4] = { v.x, v.y, v.z, v.w };
            // sixteen plain bases (A C G T in either case: 99 % of a genome) are packed four at a time without looking
            // at single bytes; anything else takes the symbol-by-symbol path
            uint32_t c0, c1, c2, c3, x0, x1, x2, x3;
            codes_of_word(w[0], c0, x0); codes_of_word(w[1], c1, x1); codes_of_word(w[2], c2, x2); codes_of_word(w[3], c3, x3);
            if ((x0 | x1 | x2 | x3) == 0u) grp = (uint64_t)(c0 | (c1 << 8) | (c2 << 16) | (c3 << 24));       // classes 0
            else grp = pack_group([&](int j) { return (uint8_t)(w[j >> 2] >> (8 * (j & 3))); }, 16, &om, &nul);
        } else {
            const uint8_t *p = A.src + b0;
            grp = pack_group([&](int j) { return p[j]; }, nv, &om, &nul);
        }
        A.dst[gi] = grp;
        if (nul) atomicOr(A.flags, 1u);
        while (om) {
            const int j = __ffs((int)om) - 1;
            om &= om - 1;
            const unsigned long long slot = atomicAdd(A.exc_n, 1ull);
            if (slot < A.exc_cap) {
                A.exc_pos[slot] = A.gbase + b0 + (uint64_t)j;
                A.exc_chr[slot] = upper_c(A.src[b0 + j]);
            }
        }
    }
}

// ===========================================================================
// K5  genome k-mer spectrum
// ===========================================================================
// One thread per packed group: the 16 k-mers that START in the group (they
// reach at most 13 bases into the next one).  K-mers touching a non-ACGT
// symbol -- which includes the padding between contigs, so no k-mer spans two
// contigs (genome-kmer-count.c:56-58) -- are skipped (kmer.c:94-96,207-208).
constexpr int kSpectrumSmemK = 6;     // 4^6 u32 bins = 16 KB privatised per CTA

// CT = counter type of the global table: unsigned int while the genome has fewer than 2^32 positions (no bin can
// overflow; 4^12 bins are then 64 MiB and stay in L2), unsigned long long otherwise.
template <bool SMEM, typename CT>
__global__ void __launch_bounds__(256) spectrum_kernel(const uint64_t *__restrict__ groups, uint64_t g_begin, uint64_t g_end,
                                                       int K, CT *__restrict__ counts)
{
    __shared__ uint32_t s_hist[SMEM ? (1 << (2 * kSpectrumSmemK)) : 1];
    const uint32_t n_bins = 1u << (2 * K);
    if (SMEM) {
        for (uint32_t i = threadIdx.x; i < n_bins; i += blockDim.x) s_hist[i] = 0;
        __syncthreads();
    }
    const uint32_t kmask = n_bins - 1u;
    const uint64_t kmask64 = kmask;
    for (uint64_t gi = g_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; gi < g_end;
         gi += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t g0 = __ldg(groups + gi), g1 = __ldg(groups + gi + 1);
        const uint64_t codes = (uint64_t)(uint32_t)g0 | ((uint64_t)(uint32_t)g1 << 32);
        const uint64_t cls = (g0 >> 32) | (g1 & 0xffffffff00000000ull);
        const uint64_t bad = (cls | (cls >> 1)) & kEvenBits;
        if ((uint32_t)bad == 0x55555555u) continue;          // whole group invalid (padding / N run)
#pragma unroll
        for (int o = 0; o < 16; o++) {
            if (((bad >> (2 * o)) & kmask64) != 0) continue;
            const uint32_t w = (uint32_t)(codes >> (2 * o)) & kmask;
            const uint32_t idx = rev_fields32(w) >> (32 - 2 * K);
            if (SMEM) atomicAdd(&s_hist[idx], 1u);
            else      atomicAdd(counts + idx, (CT)1);
        }
    }
    if (SMEM) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n_bins; i += blockDim.x) {
            const uint32_t v = s_hist[i];
            if (v) atomicAdd(counts + i, (CT)v);
        }
    }
}
// k = 7 .. 9: privatised in shared memory.  The global-atomic kernel above spends 21 ms on the 3.1 Gb genome at k = 8
// (65 536 hot bins in L2, 185 G atomics/s); counting with shared-memory atomics instead is bound by instruction issue.
// Each CTA (slice, pass) counts the k-mers of its slice whose index falls into the pass's bin range and adds its bins
// to the global table once.  The window is turned MSB-first once, so a k-mer index is one shift and one mask
// (kmer.c:184-214 order).
constexpr int kSpecSmemLog  = 15;
constexpr int kSpecSmemBins = 1 << kSpecSmemLog;
constexpr int kSpecSmemThreads = 1024;
// 65 536 bins per pass in 128 KB of shared memory, as 16-bit counters packed two to a word -- bin b lives in half
// (b >> 15) & 1 of word b & 0x7fff -- so 4^8 bins take ONE pass over the packed genome (0.25 ms from HBM), with no pass
// test in the per-k-mer code, and 4^9 take four.  A 16-bit counter cannot hold a hot bin
// (poly-A: 10^8 hits), so it is drained on the fly, exactly: an increment is a 32-bit shared-memory atomic add of 1 or
// 0x10000 that returns the old word; the old words of a group's 16 increments are OR-ed and looked at once -- if some
// half had reached 0x8000, the thread clears that bit with an atomicAnd and, if it was the one that cleared it, adds
// 32 768 to the global bin.  Between a half reaching 0x8000 and the first drain at most 16 increments per thread of the
// CTA arrive (16 384 < 0x8000): a half never wraps and never carries into its neighbour.  k-mer validity (all K bases
// ACGT) comes from one smeared mask per group, and a group without a bad base (99 % of them) runs 16 unpredicated
// increments.
constexpr int kSpec16Log   = 16;                   // bins per pass
constexpr int kSpec16Words = 1 << 15;              // 32-bit words of shared memory
template <int K, int NPASS, bool ALL, typename CT>
__device__ __forceinline__ void spec16_group(uint32_t *s_words, uint64_t msb, uint32_t vmask, uint32_t pass, CT *__restrict__ counts)
{
    constexpr uint32_t n_bins = 1u << (2 * K);
    constexpr uint32_t kmask = n_bins - 1u;
    uint32_t acc = 0;
#pragma unroll
    for (int o = 0; o < 16; o++) {
        if (!ALL && !((vmask >> (2 * o)) & 1u)) continue;
        const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & kmask;
        if (NPASS > 1 && (idx >> kSpec16Log) != pass) continue;
        const uint32_t inc = (2 * K > 15) ? ((idx >> 15) & 1u) * 0xffffu + 1u : 1u;
        acc |= atomicAdd(&s_words[idx & 0x7fffu], inc);
    }
    if (acc & 0x80008000u) {                       // rare: some half is past 0x8000 -- drain what this thread touched
#pragma unroll 1
        for (int o = 0; o < 16; o++) {
            if (!ALL && !((vmask >> (2 * o)) & 1u)) continue;
            const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & kmask;
            if (NPASS > 1 && (idx >> kSpec16Log) != pass) continue;
            const uint32_t bit = ((idx >> 15) & 1u) ? 0x80000000u : 0x8000u;
            if (atomicAnd(&s_words[idx & 0x7fffu], ~bit) & bit) atomicAdd(counts + idx, (CT)32768);
        }
    }
}
// the same for a group of low-complexity sequence: per k-mer, the lanes of the warp that are here and want the same bin
// elect one that adds for all (an increment of at most 32 per atomic: the drain bound of 16 increments per thread holds)
template <int K, int NPASS, typename CT>
__device__ __noinline__ void spec16_group_aggregated(uint32_t *s_words, uint64_t msb, uint32_t vmask, uint32_t pass, CT *__restrict__ counts)
{
    constexpr uint32_t n_bins = 1u << (2 * K);
    constexpr uint32_t kmask = n_bins - 1u;
    const uint32_t here = __activemask(), lane = threadIdx.x & 31u;
    uint32_t acc = 0;
#pragma unroll 1
    for (int o = 0; o < 16; o++) {
        const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & kmask;
        const bool     want = ((vmask >> (2 * o)) & 1u) && (NPASS == 1 || (idx >> kSpec16Log) == pass);
        // lanes that do not count this k-mer get a key of their own (bit 31 + lane) and add nothing
        const uint32_t peers = __match_any_sync(here, want ? idx : (0x80000000u | lane));
        if (want && lane == (uint32_t)__ffs((int)peers) - 1u) {
            const uint32_t inc = (2 * K > 15) ? ((idx >> 15) & 1u) * 0xffffu + 1u : 1u;
            acc |= atomicAdd(&s_words[idx & 0x7fffu], inc * (uint32_t)__popc(peers));
        }
    }
    if (acc & 0x80008000u) {
#pragma unroll 1
        for (int o = 0; o < 16; o++) {
            if (!((vmask >> (2 * o)) & 1u)) continue;
            const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & kmask;
            if (NPASS > 1 && (idx >> kSpec16Log) != pass) continue;
            const uint32_t bit = ((idx >> 15) & 1u) ? 0x80000000u : 0x8000u;
            if (atomicAnd(&s_words[idx & 0x7fffu], ~bit) & bit) atomicAdd(counts + idx, (CT)32768);
        }
    }
}
template <int K, typename CT>
__global__ void __launch_bounds__(kSpecSmemThreads, 1) spectrum_smem16_kernel(const uint64_t *__restrict__ groups, uint64_t g_begin,
                                                                               uint64_t g_end, uint32_t n_slices, CT *__restrict__ counts)
{
    extern __shared__ uint32_t s_words[];
    constexpr uint32_t n_bins = 1u << (2 * K);
    constexpr int      NPASS = n_bins > (1u << kSpec16Log) ? (int)(n_bins >> kSpec16Log) : 1;
    constexpr uint32_t words = n_bins >= (1u << kSpec16Log) ? (uint32_t)kSpec16Words : (n_bins > 32768u ? 32768u : n_bins);
    const uint32_t slice = blockIdx.x % n_slices, pass = blockIdx.x / n_slices;
    for (uint32_t i = threadIdx.x; i < words; i += kSpecSmemThreads) s_words[i] = 0;
    __syncthreads();
    const uint64_t n = g_end - g_begin;
    const uint64_t lo = g_begin + n * slice / n_slices, hi = g_begin + n * (slice + 1) / n_slices;
    for (uint64_t gi = lo + threadIdx.x; gi < hi; gi += kSpecSmemThreads) {
        const uint64_t g0 = __ldg(groups + gi), g1 = __ldg(groups + gi + 1);
        const uint64_t cls = (g0 >> 32) | (g1 & 0xffffffff00000000ull);
        uint64_t       bad = (cls | (cls >> 1)) & kEvenBits;                 // bit 2j: base j of the 32-base window is not ACGT
        if ((uint32_t)bad == 0x55555555u) continue;                          // whole group invalid (padding / N run)
        const uint64_t codes = (uint64_t)(uint32_t)g0 | ((uint64_t)(uint32_t)g1 << 32);
        const uint64_t msb = rev_fields64(codes, 32);                        // base j of the window at field 31 - j
        // smear: bit 2o set <=> some base of [o, o + K) is bad
        {
            int span = 1;
#pragma unroll
            for (int it = 0; it < 4; it++) {
                const int step = span < K - span ? span : K - span;
                if (step > 0) { bad |= bad >> (2 * step); span += step; }
            }
        }
        const uint32_t inval = (uint32_t)bad & 0x55555555u;
        // Low-complexity sequence (poly-A, (CA)n, (CAG)n ...): the window repeats with period 2 or 3 (a homopolymer with
        // both), every lane of the warp then asks for the same few bins and the shared-memory atomics would serialise
        // 32 ways.  Such groups take a path in which the lanes that want the same bin are found with match.any and one
        // of them adds the popcount.
        const bool periodic = ((msb ^ (msb >> 4)) << 4) == 0ull || ((msb ^ (msb >> 6)) << 6) == 0ull;
        if (periodic) spec16_group_aggregated<K, NPASS, CT>(s_words, msb, ~inval, pass, counts);
        else if (inval == 0u) spec16_group<K, NPASS, true, CT>(s_words, msb, 0u, pass, counts);
        else spec16_group<K, NPASS, false, CT>(s_words, msb, ~inval, pass, counts);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < words; i += kSpecSmemThreads) {
        const uint32_t v = s_words[i], lo16 = v & 0xffffu, hi16 = v >> 16;
        const size_t   base = (size_t)pass << kSpec16Log;
        if (lo16) atomicAdd(counts + base + i, (CT)lo16);
        if (hi16) atomicAdd(counts + base + 0x8000u + i, (CT)hi16);
    }
}
// k = 10 .. 12: one global atomic per k-mer is bound by the rate at which the SMs can send requests to L2 (16 ms for the
// 3.1 Gb genome, 4^12 bins resident in L2).  Instead: (1) count the k-mers per bucket = high 2k-15 bits of the index
// (<= 512 buckets), (2) scatter the low 15 bits of every k-mer, as u16, into its bucket's stretch of a scratch buffer
// -- tile by tile, a tile's k-mers sorted by bucket in shared memory first, so that a bucket needs one global atomic
// per tile and the stores leave in runs -- (3) per bucket, a 32 768-bin histogram in shared memory.  32 bytes of
// scratch per packed group; the k-mers cross HBM twice (2 bytes each) instead of crossing the L2 atomics once.
constexpr int kRadixThreads = 512;                            // = groups per tile = most buckets
// bit 2o of the result set <=> the k-mer that starts at base o of the window touches a base that is not ACGT
template <int K>
__device__ __forceinline__ uint32_t smear_bad(uint64_t bad)
{
    int span = 1;
#pragma unroll
    for (int it = 0; it < 4; it++) {
        const int step = span < K - span ? span : K - span;
        if (step > 0) { bad |= bad >> (2 * step); span += step; }
    }
    return (uint32_t)bad & 0x55555555u;
}
template <int K>
__device__ __forceinline__ bool radix_kmers(const uint64_t *__restrict__ groups, uint64_t gi, uint64_t &msb, uint64_t &bad)
{
    const uint64_t g0 = __ldg(groups + gi), g1 = __ldg(groups + gi + 1);
    const uint64_t codes = (uint64_t)(uint32_t)g0 | ((uint64_t)(uint32_t)g1 << 32);
    const uint64_t cls = (g0 >> 32) | (g1 & 0xffffffff00000000ull);
    bad = (cls | (cls >> 1)) & kEvenBits;
    msb = rev_fields64(codes, 32);
    return (uint32_t)bad != 0x55555555u;
}
template <int K>
__global__ void __launch_bounds__(kRadixThreads) radix_count_kernel(const uint64_t *__restrict__ groups, uint64_t g_begin, uint64_t g_end,
                                                                     unsigned long long *__restrict__ bucket_cnt)
{
    constexpr uint32_t nb = 1u << (2 * K - kSpecSmemLog);
    constexpr uint64_t kmask = (1ull << (2 * K)) - 1ull;
    __shared__ uint32_t s_cnt[nb];
    for (uint32_t i = threadIdx.x; i < nb; i += kRadixThreads) s_cnt[i] = 0;
    __syncthreads();
    for (uint64_t gi = g_begin + (uint64_t)blockIdx.x * kRadixThreads + threadIdx.x; gi < g_end; gi += (uint64_t)gridDim.x * kRadixThreads) {
        uint64_t msb, bad;
        if (!radix_kmers<K>(groups, gi, msb, bad)) continue;
        const uint32_t inval = smear_bad<K>(bad);
#pragma unroll
        for (int o = 0; o < 16; o++) {
            if ((inval >> (2 * o)) & 1u) continue;
            const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & (uint32_t)kmask;
            atomicAdd(&s_cnt[idx >> kSpecSmemLog], 1u);
        }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nb; i += kRadixThreads)
        if (s_cnt[i]) atomicAdd(bucket_cnt + i, (unsigned long long)s_cnt[i]);
}
// exclusive scan of the bucket counts (one block): off[0..nb], cursor[b] = off[b]
__global__ void __launch_bounds__(kRadixThreads) radix_scan_kernel(const unsigned long long *__restrict__ cnt, unsigned long long *__restrict__ off,
                                                                    unsigned long long *__restrict__ cursor, uint32_t nb)
{
    __shared__ unsigned long long s[kRadixThreads];
    const uint32_t t = threadIdx.x;
    s[t] = t < nb ? cnt[t] : 0ull;
    __syncthreads();
    for (uint32_t d = 1; d < kRadixThreads; d <<= 1) {
        const unsigned long long v = t >= d ? s[t - d] : 0ull;
        __syncthreads();
        s[t] += v;
        __syncthreads();
    }
    if (t < nb) { const unsigned long long ex = s[t] - cnt[t]; off[t] = ex; cursor[t] = ex; }
    if (t == nb - 1) off[nb] = s[t];
}
template <int K>
__global__ void __launch_bounds__(kRadixThreads) radix_scatter_kernel(const uint64_t *__restrict__ groups, uint64_t g_begin, uint64_t g_end,
                                                                       unsigned long long *__restrict__ cursor, uint16_t *__restrict__ payload)
{
    constexpr uint32_t nb = 1u << (2 * K - kSpecSmemLog);
    constexpr uint64_t kmask = (1ull << (2 * K)) - 1ull;
    __shared__ uint32_t s_cnt[kRadixThreads], s_toff[kRadixThreads + 1], s_warp[kRadixThreads / 32];
    __shared__ unsigned long long s_goff[kRadixThreads];
    __shared__ uint32_t s_rec[16 * kRadixThreads];            // payload | bucket << 16, in bucket order: one store per k-mer
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    const uint64_t n_tiles = (g_end - g_begin + kRadixThreads - 1) / kRadixThreads;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t gi = g_begin + tile * kRadixThreads + t;
        s_cnt[t] = 0;
        __syncthreads();
        uint64_t msb = 0, bad = ~0ull;
        const bool any = gi < g_end && radix_kmers<K>(groups, gi, msb, bad);
        // bucket and rank within (tile, bucket) of each of the 16 k-mers, kept in registers for the second step
        uint32_t br[16];
        uint32_t vm = 0;
        if (any) {
            const uint32_t inval = smear_bad<K>(bad);
#pragma unroll
            for (int o = 0; o < 16; o++) {
                br[o] = 0;
                if ((inval >> (2 * o)) & 1u) continue;
                const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & (uint32_t)kmask;
                const uint32_t b = idx >> kSpecSmemLog;
                br[o] = b | (atomicAdd(&s_cnt[b], 1u) << 9);
                vm |= 1u << o;
            }
        }
        __syncthreads();
        // exclusive scan of the per-bucket counts of this tile (t = bucket); global stretch for each bucket
        const uint32_t c = t < nb ? s_cnt[t] : 0u;
        uint32_t inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
            if ((int)lane >= d) inc += v;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        uint32_t base = 0;
        for (uint32_t w = 0; w < warp; w++) base += s_warp[w];
        s_toff[t] = base + inc - c;
        if (t == kRadixThreads - 1) s_toff[kRadixThreads] = base + inc;
        if (c) s_goff[t] = atomicAdd(cursor + t, (unsigned long long)c) - (unsigned long long)(base + inc - c);   // global - tile offset
        __syncthreads();
        if (vm) {
#pragma unroll
            for (int o = 0; o < 16; o++) {
                if (!((vm >> o) & 1u)) continue;
                const uint32_t idx = (uint32_t)(msb >> (2 * (32 - o - K))) & (uint32_t)kmask;
                const uint32_t b = br[o] & 511u;
                const uint32_t pos = s_toff[b] + (br[o] >> 9);
                s_rec[pos] = (idx & (uint32_t)(kSpecSmemBins - 1)) | (b << 16);
            }
        }
        __syncthreads();
        const uint32_t n_tile = s_toff[kRadixThreads];
        for (uint32_t i = t; i < n_tile; i += kRadixThreads) { const uint32_t v = s_rec[i]; payload[s_goff[v >> 16] + i] = (uint16_t)v; }
        __syncthreads();
    }
}
// bucket (blockIdx.x / parts), part (blockIdx.x % parts): 32 768-bin shared-memory histogram of a stretch of payloads
template <typename CT>
__global__ void __launch_bounds__(kSpecSmemThreads, 1) radix_hist_kernel(const uint16_t *__restrict__ payload, const unsigned long long *__restrict__ off,
                                                                          uint32_t parts, CT *__restrict__ counts)
{
    extern __shared__ uint32_t s_bins[];
    const uint32_t b = blockIdx.x / parts, part = blockIdx.x % parts;
    for (uint32_t i = threadIdx.x; i < (uint32_t)kSpecSmemBins; i += kSpecSmemThreads) s_bins[i] = 0;
    __syncthreads();
    const unsigned long long lo0 = off[b], n = off[b + 1] - lo0;
    const unsigned long long lo = lo0 + n * part / parts, hi = lo0 + n * (part + 1) / parts;
    // head up to a 16-byte boundary, body as uint4 (8 payloads), tail
    unsigned long long a = (lo + 7ull) & ~7ull;
    if (a > hi) a = hi;
    for (unsigned long long i = lo + threadIdx.x; i < a; i += kSpecSmemThreads) atomicAdd(&s_bins[payload[i]], 1u);
    const unsigned long long body = (hi - a) / 8;
    const uint4 *p4 = reinterpret_cast<const uint4 *>(payload + a);
    for (unsigned long long i = threadIdx.x; i < body; i += kSpecSmemThreads) {
        const uint4 v = __ldg(p4 + i);
        atomicAdd(&s_bins[v.x & 0xffffu], 1u); atomicAdd(&s_bins[v.x >> 16], 1u);
        atomicAdd(&s_bins[v.y & 0xffffu], 1u); atomicAdd(&s_bins[v.y >> 16], 1u);
        atomicAdd(&s_bins[v.z & 0xffffu], 1u); atomicAdd(&s_bins[v.z >> 16], 1u);
        atomicAdd(&s_bins[v.w & 0xffffu], 1u); atomicAdd(&s_bins[v.w >> 16], 1u);
    }
    for (unsigned long long i = a + body * 8 + threadIdx.x; i < hi; i += kSpecSmemThreads) atomicAdd(&s_bins[payload[i]], 1u);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < (uint32_t)kSpecSmemBins; i += kSpecSmemThreads) {
        const uint32_t v = s_bins[i];
        if (v) atomicAdd(counts + ((size_t)b << kSpecSmemLog) + i, (CT)v);
    }
}
// (Measured and rejected, round 2: a "write combining" partition -- per-warp 32-byte buffers per bucket in shared
// memory, appended with shared-memory atomics, flushed by the lane that fills one -- is exact but three times slower
// than the in-tile sort above (38 ms against 12 ms at k = 12, 103 ms against 10 ms at k = 10 with its 16 buckets): every
// flush needs a global atomic on the bucket's cursor and the whole warp waits for it at the next __syncwarp, about twice
// per round of 32 k-mers.  profiles/r2_spectrum_radix_write_combining_experiment.json; git history has the kernels.)
// u32 spectrum -> u64 output
__global__ void __launch_bounds__(256) widen_kernel(const unsigned int *__restrict__ in, unsigned long long *__restrict__ out, uint64_t n)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) out[i] = in[i];
}

// ===========================================================================
// K1-K4  SAM tile scan + per-record tally
// ===========================================================================
// measured best: 2 CTAs of 256 threads per SM, 4 scan steps per tile
constexpr int kCtasPerSm  = 2;
constexpr int kThreads    = 256;                              // threads per CTA = records a CTA takes per tile
constexpr int kWarps      = kThreads / 32;
constexpr int kIters      = 4;                                // steps of the scan
constexpr int kSlots      = kIters * kThreads;                // 64-byte slots (two 32-byte chunks) of one tile
constexpr int kChunks     = 2 * kSlots;                       // chunks = mask words of one tile
constexpr int kSpan       = kChunks * 32;                     // bytes of staged text
constexpr int kPrefix     = 16;                               // the bulk copy lands at bytes + kPrefix; the byte before the first
                                                              // record (a '\n') sits in [kPrefix - 1, 2 * kPrefix)
constexpr int kStageMax   = kSpan - 80;                       // most bytes of one bulk copy: the data always ends below kSpan - 64
constexpr int kSegs       = kIters * kWarps;                  // warp-iterations of the scan = segments of the newline ranking
constexpr int kCacheContigs = 64;                             // contig table kept in shared memory when it fits
constexpr int kCacheNames   = 1024;
constexpr int kCacheSlots   = 1024;                          // u8 slots of the collision-free name table
constexpr int kFlushEvery   = 1900;                           // warp iterations between flushes of the 16-bit partial sums
static_assert(kThreads % 32 == 0 && kSlots % 32 == 0 && kSegs <= 64, "the newline ranking keeps at most two segment counts per lane");
static_assert(kThreads >= kCacheContigs, "one thread per cached contig fills the shared-memory table");
static_assert(kSpan < (1 << 20) && kThreads <= 1024, "pass A packs a newline position into 20 bits and its rank into the rest");

struct ContigCache {
    uint32_t n;                                               // 0: not cached, use the global table
    uint32_t seed;                                            // the host found it: no two names share a slot
    uint16_t name_w0[kCacheContigs], name_len[kCacheContigs]; // first word of the name in names32 / length in bytes
    uint64_t base_off[kCacheContigs], len[kCacheContigs];
    uint8_t  slot[kCacheSlots];                               // slot -> contig, 0xff = empty
    uint32_t names32[kCacheNames / 4 + 2 * kCacheContigs];    // names as zero-padded little-endian words, one spare word each
};

struct TallyShared {                                          // per-CTA tables, outcome counters, contig table
    uint32_t table[2 * 32 * 16];                              // CTA count tables [fwd|rev][row][cell]
    uint32_t stats[8];                                        // outcomes (pss-bam's in the fused mode)
    uint32_t stats_fk[8];                                     // fragkon's outcomes in the fused mode
    ContigCache cc;
};

struct TallySmem {
    alignas(128) uint8_t bytes[kSpan + 32];                   // staged SAM text (+ slack for word reads past the last record)
    alignas(8) uint32_t le[kChunks + 8];                      // bit i of word c: byte 32c+i is <= 0x20; 8 all-ones sentinels
    uint32_t seg[64];                                         // per segment (one warp-iteration of the scan): which chunks hold a newline
    uint32_t nlpos[kThreads + 4];                             // positions of the first kThreads + 1 newlines
    uint32_t warp_sum[kWarps];                                // generic newline listing only
    uint32_t ctl[2];                                          // range handed to this CTA
    uint32_t text_done;                                       // warps done reading a tile's text (a multiple of kWarps
                                                              // between tiles that copy the next one early)
    unsigned long long long_end;                              // where a record longer than the tile ends
    TallyShared sh;
    alignas(8) uint64_t bar;
};

struct TallyArgs {
    const uint8_t *sam;          // device, 16-byte aligned
    uint64_t       len;          // bytes of text (an upper bound when len_dev is set)
    const unsigned long long *len_dev;   // non-null: the length is read from device memory when the kernel starts (text produced
                                         // by an earlier kernel of the stream, e.g. the BAM renderer)
    uint64_t       stream_off;   // offset of sam[0] within everything fed (debug log only)
    uint64_t       range_bytes;  // the text is handed out in ranges of this many bytes (multiple of 32)
    unsigned int  *range_ctr;    // next range (zero before the launch)
    uint32_t       one;          // 1, opaque to the compiler: turns additions into IMADs (FMA pipe) where the ALU pipe is the limit
    DevGenome      g;
    TallyCfg       cfg;          // pss-bam options (fragkon's when only fragkon runs)
    TallyCfg       cfg_fk;       // fragkon options of the fused mode
    uint32_t       names_bytes;  // total bytes of contig names
    uint32_t       cc_seed;      // seed of the collision-free hash of the contig names ...
    uint32_t       cc_ok;        // ... if the host found one (<= kCacheContigs names of <= kCacheNames bytes)
    unsigned long long *pss_tables;   // 2*(R+2)*16 u64: fwd then rev
    unsigned long long *fk_hist;      // 2*4^K u64: 5' then 3'
    unsigned long long *stats;        // kStN
    unsigned long long *stats_fk;     // kStN, fused mode only
    uint64_t           *dbg_off;      // debug log (may be null)
    int8_t             *dbg_code;
    unsigned long long *dbg_n;
    uint64_t            dbg_cap;
};

struct SmemAt {                  // absolute positions in the staged tile (4-byte aligned base)
    static constexpr int kLookBack = kPrefix;       // every record starts at >= kPrefix: 12 bytes back is always inside
    const uint8_t *p;
    __device__ __forceinline__ int lo() const { return 0; }
    __device__ __forceinline__ uint32_t operator()(int i) const { return p[i]; }
    __device__ __forceinline__ uint32_t word(int i) const { return *reinterpret_cast<const uint32_t *>(p + i); }
};
struct SmemRel {                 // positions relative to a record start (any alignment); records start at >= kPrefix
    static constexpr int kLookBack = kPrefix;
    const uint8_t *p;
    __device__ __forceinline__ int lo() const { return -kPrefix; }
    __device__ __forceinline__ uint32_t operator()(int i) const { return p[i]; }
    __device__ __forceinline__ uint32_t word(int i) const
    {
        return (uint32_t)p[i] | ((uint32_t)p[i + 1] << 8) | ((uint32_t)p[i + 2] << 16) | ((uint32_t)p[i + 3] << 24);
    }
};
struct GlobalAt {                // positions relative to p; nothing before p is touched
    static constexpr int kLookBack = 0;
    const uint8_t *p;
    __device__ __forceinline__ int lo() const { return 0; }
    __device__ __forceinline__ uint32_t operator()(int i) const { return __ldg(p + i); }
    __device__ __forceinline__ uint32_t word(int i) const
    {
        return (uint32_t)__ldg(p + i) | ((uint32_t)__ldg(p + i + 1) << 8) | ((uint32_t)__ldg(p + i + 2) << 16) |
               ((uint32_t)__ldg(p + i + 3) << 24);
    }
};

// LOP3 / IMAD spelled out: the compiler's canonical forms of these expressions cost an extra instruction per word
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return d;
}
__device__ __forceinline__ uint32_t imad(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// 0x80 in every byte of w that is <= 0x20 / that is '\n'.  Three ALU-pipe and three FMA-pipe instructions per word:
// `one` is 1 at run time but a kernel argument, so opaque to the compiler: the additions are issued as IMADs (the
// kernel is bound by the integer ALU pipe, the FMA pipe is otherwise idle).  On the low seven bits v of a byte, bit 7
// of v + (0x80 - k) says v >= k; a byte is <= 0x20 when its bit 7 is clear and v < 0x21, and '\n' when, in addition,
// v >= 0x0a and v < 0x0b.
__device__ __forceinline__ void classify4(uint32_t w, uint32_t one, uint32_t &zle, uint32_t &znl)
{
    const uint32_t v = w & 0x7f7f7f7fu;
    const uint32_t ge21 = imad(v, one, 0x5f5f5f5fu);
    const uint32_t ge0a = imad(v, one, 0x76767676u);
    const uint32_t ge0b = imad(v, one, 0x75757575u);
    zle = lop3<0x02>(ge21, w, 0x80808080u);                             // ~(ge21 | w) & 0x80808080
    znl = lop3<0x20>(zle, ge0b, ge0a);                                  // zle & ~ge0b & ge0a
}
// The scan's variant: the "<= 0x20" flags as above, and instead of the exact newline flags just bit 1 of every byte
// (one AND).  '\n' = 0x0a has it, '\t' = 0x09 and ' ' = 0x20 do not: "<= 0x20 and bit 1" finds every newline plus
// a few control bytes that real text does not contain; pass A checks each candidate against the byte itself and
// sends a tile with a false one to the exact listing.  Three ALU-pipe + one FMA-pipe instruction per word.
__device__ __forceinline__ void classify4_fast(uint32_t w, uint32_t one, uint32_t &zle, uint32_t &p1)
{
    const uint32_t v = w & 0x7f7f7f7fu;
    const uint32_t ge21 = imad(v, one, 0x5f5f5f5fu);
    zle = lop3<0x02>(ge21, w, 0x80808080u);                             // ~(ge21 | w) & 0x80808080
    p1 = w & 0x02020202u;
}
// 8 flag bytes (0x80 / 0) in two words -> 8-bit mask << 7, via two byte dot products
__device__ __forceinline__ uint32_t gather8(uint32_t z0, uint32_t z1)
{
    return __dp4a(z1, 0x80402010u, __dp4a(z0, 0x08040201u, 0u));
}
// the two mask words of one 32-byte chunk
__device__ __forceinline__ void classify32(const uint8_t *p, uint32_t one, uint32_t &le32, uint32_t &nl32)
{
    const uint4 v0 = *reinterpret_cast<const uint4 *>(p);
    const uint4 v1 = *reinterpret_cast<const uint4 *>(p + 16);
    uint32_t zl[8], zn[8];
    classify4(v0.x, one, zl[0], zn[0]); classify4(v0.y, one, zl[1], zn[1]);
    classify4(v0.z, one, zl[2], zn[2]); classify4(v0.w, one, zl[3], zn[3]);
    classify4(v1.x, one, zl[4], zn[4]); classify4(v1.y, one, zl[5], zn[5]);
    classify4(v1.z, one, zl[6], zn[6]); classify4(v1.w, one, zl[7], zn[7]);
    // the four 8-bit groups do not overlap: sums instead of ORs, so the shifts ride on IMADs
    le32 = (gather8(zl[0], zl[1]) >> 7) + gather8(zl[2], zl[3]) * 2u + gather8(zl[4], zl[5]) * 512u + gather8(zl[6], zl[7]) * 131072u;
    nl32 = (gather8(zn[0], zn[1]) >> 7) + gather8(zn[2], zn[3]) * 2u + gather8(zn[4], zn[5]) * 512u + gather8(zn[6], zn[7]) * 131072u;
}

// one 32-byte chunk for the scan: "<= 0x20" mask word and newline-candidate mask word
__device__ __forceinline__ void classify32_fast(const uint4 &v0, const uint4 &v1, uint32_t one, uint32_t &le32, uint32_t &nc32)
{
    uint32_t zl[8], zp[8];
    classify4_fast(v0.x, one, zl[0], zp[0]); classify4_fast(v0.y, one, zl[1], zp[1]);
    classify4_fast(v0.z, one, zl[2], zp[2]); classify4_fast(v0.w, one, zl[3], zp[3]);
    classify4_fast(v1.x, one, zl[4], zp[4]); classify4_fast(v1.y, one, zl[5], zp[5]);
    classify4_fast(v1.z, one, zl[6], zp[6]); classify4_fast(v1.w, one, zl[7], zp[7]);
    le32 = (gather8(zl[0], zl[1]) >> 7) + gather8(zl[2], zl[3]) * 2u + gather8(zl[4], zl[5]) * 512u + gather8(zl[6], zl[7]) * 131072u;
    // plane flags are 0x02, not 0x80: the same dot products give the mask << 1
    const uint32_t p32 = (gather8(zp[0], zp[1]) >> 1) + gather8(zp[2], zp[3]) * 128u + gather8(zp[4], zp[5]) * 32768u
                       + gather8(zp[6], zp[7]) * 8388608u;
    nc32 = le32 & p32;
}

__device__ __forceinline__ void log_outcome(const TallyArgs &A, uint64_t goff, int code)
{
    if (A.dbg_n) {
        const unsigned long long slot = atomicAdd(A.dbg_n, 1ull);
        if (slot < A.dbg_cap) {
            A.dbg_off[slot] = A.stream_off + goff;
            A.dbg_code[slot] = (int8_t)code;
        }
    }
}
__device__ __forceinline__ int stat_slot(int code)
{
    return code == kCounted ? kStCounted : code == kNoContig ? kStNoContig : code == kFiltered ? kStFiltered
         : code == kParseFail ? kStParseFail : kStUndefined;
}

// k-th 4-byte word of the field [off, off+len), zero padded at the end
template <class B>
__device__ __forceinline__ uint32_t field_word(const B &b, int off, int len, int k)
{
    uint32_t  w = word_at(b, off + 4 * k);
    const int rem = len - 4 * k;
    if (rem < 4) w &= rem <= 0 ? 0u : ((1u << (8 * rem)) - 1u);
    return w;
}
template <class B>
__device__ __forceinline__ uint32_t name_hash_words(const B &b, int off, int len, uint32_t seed)
{
    // every name hashes at least its first two (zero padded) words: no loop for names of up to 8 bytes
    // (pssgpu.cu: host_name_hash is the same function; it searches the seed)
    uint32_t  h = seed ^ (uint32_t)len;
    const int nw = (len + 3) >> 2;
    h = (h ^ field_word(b, off, len, 0)) * 0x9E3779B1u;  h ^= h >> 15;
    h = (h ^ field_word(b, off, len, 1)) * 0x9E3779B1u;  h ^= h >> 15;
    for (int k = 2; k < nw; k++) {
        h = (h ^ field_word(b, off, len, k)) * 0x9E3779B1u;
        h ^= h >> 15;
    }
    return h;
}
// find_seq (fasta-genome-io.c:202-213) against the shared-memory copy of the
// contig table.  The hash is collision free on the contig names (the host
// searched the seed), so one probe and one whole-word comparison of RNAME
// decide, in straight-line code: the lanes of a warp do not drift apart here.
template <class B>
__device__ __forceinline__ int cache_find(const ContigCache &C, const B &b, int off, int len, uint64_t &base, uint64_t &clen)
{
    const uint32_t h = name_hash_words(b, off, len, C.seed);
    const uint32_t w0 = field_word(b, off, len, 0), w1 = field_word(b, off, len, 1);
    const uint32_t v = C.slot[h & (kCacheSlots - 1)];
    const uint32_t vv = v != 0xffu ? v : 0u;
    const uint32_t *nm = C.names32 + C.name_w0[vv];
    bool eq = (v != 0xffu) & ((int)C.name_len[vv] == len) & (nm[0] == w0 || len <= 0) & (nm[1] == w1 || len <= 4);
    if (len > 8) {                                    // long names: the remaining words
        const int nw = (len + 3) >> 2;
        for (int k = 2; eq && k < nw; k++) eq = (nm[k] == field_word(b, off, len, k));
    }
    base = eq ? C.base_off[vv] : 0;
    clen = eq ? C.len[vv] : 0;
    return eq ? (int)vv : -1;
}
template <class B>
__device__ __forceinline__ int lookup_contig(const ContigCache &C, const DevGenome &g, const B &b, int off, int len,
                                             uint64_t &base, uint64_t &clen)
{
    if (C.n) return cache_find(C, b, off, len, base, clen);
    const int ci = find_contig(g, b, off, len);
    base = ci >= 0 ? g.contigs[ci].base_off : 0;
    clen = ci >= 0 ? g.contigs[ci].len : 0;
    return ci;
}

// A record the tile cannot hold (longer than kStageMax, or longer than fgets'
// 200000-byte buffer): walked from global memory by one thread, split the way
// fgets(buf, MAX_LINE_LEN+1) splits it (pss-bam.c:761-764), counted with
// shared-memory atomics.  Returns the offset of the byte after the record.
// Rare by construction.
template <int MODE>
__device__ __noinline__ uint64_t long_record(const TallyArgs *Ap, TallyShared *Sp, uint64_t gstart, uint64_t text_len)
{
    const TallyArgs &A = *Ap;
    TallyShared     &S = *Sp;
    uint64_t p = gstart;
    while (p < text_len && __ldg(A.sam + p) != '\n') p++;
    uint64_t total = p - gstart + (p < text_len ? 1u : 0u);
    const uint64_t g_end = gstart + total;
    uint64_t c0 = gstart;
    while (total > 0) {
        const int L = total > (uint64_t)kMaxLine ? kMaxLine : (int)total;
        const GlobalAt at{ A.sam + c0 };
        RecView r;
        int code = scan11(at, L, r);
        if (code == kCounted) {
            uint64_t  cb, cl;
            const int ci = lookup_contig(S.cc, A.g, at, r.rname_off, r.rname_len, cb, cl);
            int code_fk = kFiltered;
            if (MODE != kModePss) {
                FkHits h;
                const TallyCfg &F = (MODE == kModeBoth) ? A.cfg_fk : A.cfg;
                code_fk = fk_record(at, r, true, ci, cb, cl, A.g, F, h);
                if (h.add5) atomicAdd(A.fk_hist + h.idx5, 1ull);
                if (h.add3) atomicAdd(A.fk_hist + (1ull << (2 * F.K)) + h.idx3, 1ull);
                if (MODE == kModeBoth) atomicAdd(&S.stats_fk[stat_slot(code_fk)], 1u);
            }
            if (MODE != kModeFragkon && A.cfg.R > kMaxRegion) {
                const int rows = A.cfg.R + 2;
                code = pss_record_wide(at, r, ci, cb, cl, A.g, A.cfg, [&](int tb, int row, int cell) {
                    atomicAdd(A.pss_tables + ((size_t)tb * rows + row) * 16 + cell, 1ull);
                });
            } else if (MODE != kModeFragkon) {
                PssStreams st;
                code = pss_record(at, r, true, ci, cb, cl, A.g, A.cfg, st);
                if (code == kCounted) {
                    const int rows = A.cfg.R + 2;
                    for (int j = 0; j < rows; j++) {
                        if (!((st.a_bad >> (2 * j)) & 1u))
                            atomicAdd(&S.table[j * 16 + (int)(((st.a_read >> (2 * j)) & 3u) * 4 + ((st.a_ref >> (2 * j)) & 3u))], 1u);
                        if (!((st.b_bad >> (2 * j)) & 1u))
                            atomicAdd(&S.table[512 + j * 16 + (int)(((st.b_read >> (2 * j)) & 3u) * 4 + ((st.b_ref >> (2 * j)) & 3u))], 1u);
                    }
                }
            } else {
                code = code_fk;
            }
        } else if (MODE == kModeBoth) {
            atomicAdd(&S.stats_fk[stat_slot(code)], 1u);      // a line that does not parse fails for both programs
        }
        atomicAdd(&S.stats[kStLines], 1u);
        if (MODE == kModeBoth) atomicAdd(&S.stats_fk[kStLines], 1u);
        atomicAdd(&S.stats[stat_slot(code)], 1u);
        log_outcome(A, c0, code);
        c0 += (uint64_t)L;
        total -= (uint64_t)L;
    }
    return g_end;
}

// ballot of "(word & mask) != 0" over the full warp: one LOP3-with-predicate + one VOTE
__device__ __forceinline__ uint32_t ballot_bits(uint32_t word, uint32_t mask)
{
    uint32_t r;
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\t"
                 "vote.sync.ballot.b32 %0, p, 0xffffffff;\n\t}" : "=r"(r) : "r"(word), "r"(mask));
    return r;
}

// ---------------------------------------------------------------------------
// The two count tables of one warp-load of records, without atomics.
//
// What a record adds is 5 bits per table and row (two bits of reference code, two of read code, "counts").  Round 1
// fetched every one of the 2 x 17 x 5 bit planes with its own ballot (LOP3 + VOTE, then IMAD picks: 37 instructions
// per row); now the warp TRANSPOSES them: five 32 x 32 bit-matrix transposes across the lanes (SHFL + PRMT for the
// byte-granular steps, SHFL + SHF + LOP3 below that: 13 instructions each) hand lane 2r + t the five planes -- one bit
// per record of the warp-load -- of row r of table t, and the lane counts its 16 cells with 20 LOP3 + 16 POPC into
// eight registers of packed 16-bit sums.  About 140 instructions per 16 rows of both tables instead of 590.
// Rows 16 and 17 (-r 15 has 17 rows) still go the ballot way: lane l owns cell (l & 15) of table (l >> 4).
// All 32 lanes must be converged.
// ---------------------------------------------------------------------------
struct XposeConsts {
    uint32_t sel16, sel8, s4, s2, s1, r4, r2, r1;
};
__device__ __forceinline__ XposeConsts xpose_consts(uint32_t lane)
{
    XposeConsts c;
    c.sel16 = (lane & 16u) ? 0x3276u : 0x5410u;
    c.sel8 = (lane & 8u) ? 0x3715u : 0x6240u;
    c.s4 = (lane & 4u) ? 0xf0f0f0f0u : 0x0f0f0f0fu;  c.r4 = (lane & 4u) ? 28u : 4u;
    c.s2 = (lane & 2u) ? 0xccccccccu : 0x33333333u;  c.r2 = (lane & 2u) ? 30u : 2u;
    c.s1 = (lane & 1u) ? 0xaaaaaaaau : 0x55555555u;  c.r1 = (lane & 1u) ? 31u : 1u;
    return c;
}
// bit j of lane i's word <-> bit i of lane j's word.  One step per bit of the index: the lower lane of a pair keeps
// the positions whose index bit is clear and takes its partner's into the others, the upper lane the other way round.
__device__ __forceinline__ uint32_t xpose32(uint32_t x, const XposeConsts &c)
{
    const uint32_t full = 0xffffffffu;
    uint32_t       t;
    t = __shfl_xor_sync(full, x, 16);  x = __byte_perm(x, t, c.sel16);
    t = __shfl_xor_sync(full, x, 8);   x = __byte_perm(x, t, c.sel8);
    t = __shfl_xor_sync(full, x, 4);   x = lop3<0xE4>(x, __funnelshift_l(t, t, c.r4), c.s4);      // (x & s) | (rot(t) & ~s)
    t = __shfl_xor_sync(full, x, 2);   x = lop3<0xE4>(x, __funnelshift_l(t, t, c.r2), c.s2);
    t = __shfl_xor_sync(full, x, 1);   x = lop3<0xE4>(x, __funnelshift_l(t, t, c.r1), c.s1);
    return x;
}
// rows [16 set, 16 set + 16) of both tables: acc[0..7] = the 16 cells of (table lane & 1, row 16 set + lane / 2)
__device__ __forceinline__ void tally_set16(uint32_t aref, uint32_t aread, uint32_t abad, uint32_t bref, uint32_t bread, uint32_t bbad,
                                            uint32_t row_mask, const XposeConsts &xc, uint32_t *acc, uint32_t one)
{
    constexpr uint32_t E = 0x55555555u;
    // bit 2r: table a, bit 2r + 1: table b -- one word per plane
    const uint32_t X0 = xpose32(lop3<0xE4>(aref, bref << 1, E), xc), X1 = xpose32(lop3<0xE4>(aref >> 1, bref, E), xc);
    const uint32_t Y0 = xpose32(lop3<0xE4>(aread, bread << 1, E), xc), Y1 = xpose32(lop3<0xE4>(aread >> 1, bread, E), xc);
    const uint32_t ga = ~abad & row_mask, gb = ~bbad & row_mask;
    const uint32_t G = xpose32(ga | (gb << 1), xc);
    uint32_t q[4];
    q[0] = lop3<0x10>(G, Y1, Y0); q[1] = lop3<0x20>(G, Y1, Y0); q[2] = lop3<0x40>(G, Y1, Y0); q[3] = lop3<0x80>(G, Y1, Y0);
#pragma unroll
    for (int k = 0; k < 4; k++) {                            // cell = read * 4 + ref (pss-bam.c:24-35)
        const uint32_t n0 = (uint32_t)__popc(lop3<0x10>(q[k], X1, X0)), n1 = (uint32_t)__popc(lop3<0x20>(q[k], X1, X0));
        const uint32_t n2 = (uint32_t)__popc(lop3<0x40>(q[k], X1, X0)), n3 = (uint32_t)__popc(lop3<0x80>(q[k], X1, X0));
        acc[2 * k] = imad(n1, 65536u, imad(n0, one, acc[2 * k]));
        acc[2 * k + 1] = imad(n3, 65536u, imad(n2, one, acc[2 * k + 1]));
    }
}
template <int NACC, int ROWS>
__device__ __forceinline__ void tally_rows(const PssStreams &st, uint32_t (&acc)[NACC ? NACC : 1], int rows, uint32_t lane, uint32_t one)
{
    static_assert(NACC == 0 || NACC == 9 || NACC == 16, "9: rows 0..15 transposed + rows 16, 17 by ballots; 16: two transposed sets");
    constexpr uint32_t E = 0x55555555u;
    const XposeConsts xc = xpose_consts(lane);
    {
        const int      n0 = ROWS ? (ROWS < 16 ? ROWS : 16) : (rows < 16 ? rows : 16);
        const uint32_t m0 = n0 >= 16 ? E : (((1u << (2 * n0)) - 1u) & E);
        tally_set16((uint32_t)st.a_ref, (uint32_t)st.a_read, (uint32_t)st.a_bad, (uint32_t)st.b_ref, (uint32_t)st.b_read, (uint32_t)st.b_bad,
                    m0, xc, acc, one);
    }
    if (NACC == 16) {
        if (rows > 16) {                                      // warp uniform
            const int      n1 = rows - 16;
            const uint32_t m1 = n1 >= 16 ? E : (((1u << (2 * n1)) - 1u) & E);
            tally_set16((uint32_t)(st.a_ref >> 32), (uint32_t)(st.a_read >> 32), (uint32_t)(st.a_bad >> 32), (uint32_t)(st.b_ref >> 32),
                        (uint32_t)(st.b_read >> 32), (uint32_t)(st.b_bad >> 32), m1, xc, acc + 8, one);
        }
        return;
    }
    constexpr int kFirstBallotRow = 16;
    const uint32_t tbi = lane >> 4;                           // which table this lane counts for
    const uint32_t neg1 = 0u - one;
    const uint32_t cell = lane & 15u;
    const uint32_t x0 = (cell & 1u) ? 0u : ~0u, x1 = (cell & 2u) ? 0u : ~0u;
    const uint32_t x2 = (cell & 4u) ? 0u : ~0u, x3 = (cell & 8u) ? 0u : ~0u;
    // "row adds nothing" flags become "row counts" flags so that every ballot is a != 0 test
    const uint32_t ar[2] = { (uint32_t)st.a_ref, (uint32_t)(st.a_ref >> 32) }, aq[2] = { (uint32_t)st.a_read, (uint32_t)(st.a_read >> 32) };
    const uint32_t ag[2] = { ~(uint32_t)st.a_bad, ~(uint32_t)(st.a_bad >> 32) };
    const uint32_t br[2] = { (uint32_t)st.b_ref, (uint32_t)(st.b_ref >> 32) }, bq[2] = { (uint32_t)st.b_read, (uint32_t)(st.b_read >> 32) };
    const uint32_t bg[2] = { ~(uint32_t)st.b_bad, ~(uint32_t)(st.b_bad >> 32) };
    // the ballots are warp uniform, the table a lane counts for is not: "tb ? b : a" as a + tb * (b - a), two IMADs
    // on the idle FMA pipe instead of a SEL on the ALU pipe (the pipe this kernel is bound by)
    auto pick = [&](uint32_t a, uint32_t b) { return imad(tbi, imad(a, neg1, b), a); };
#pragma unroll
    for (int j = kFirstBallotRow; j < 2 * NACC; j++) {
        if (ROWS ? j >= ROWS : j >= rows) break;              // ROWS: the row count as a compile-time constant (0: run time)
        const int      h = j >> 4;
        const uint32_t m0 = 1u << (2 * (j & 15)), m1 = 2u << (2 * (j & 15));
        const uint32_t a0 = ballot_bits(ar[h], m0), a1 = ballot_bits(ar[h], m1);
        const uint32_t a2 = ballot_bits(aq[h], m0), a3 = ballot_bits(aq[h], m1);
        const uint32_t av = ballot_bits(ag[h], m0);
        const uint32_t b0 = ballot_bits(br[h], m0), b1 = ballot_bits(br[h], m1);
        const uint32_t b2 = ballot_bits(bq[h], m0), b3 = ballot_bits(bq[h], m1);
        const uint32_t bv = ballot_bits(bg[h], m0);
        const uint32_t m = pick(av, bv) & (pick(a0, b0) ^ x0) & (pick(a1, b1) ^ x1) & (pick(a2, b2) ^ x2) & (pick(a3, b3) ^ x3);
        acc[j >> 1] += (uint32_t)__popc(m) << (16 * (j & 1));
    }
}
template <int NACC>
__device__ __forceinline__ void flush_acc(uint32_t (&acc)[NACC ? NACC : 1], int rows, uint32_t lane, uint32_t *table)
{
    {
        const uint32_t tb = lane & 1u, row = lane >> 1;
#pragma unroll
        for (int h = 0; h < (NACC == 16 ? 2 : 1); h++) {
            if ((int)row + 16 * h >= rows) break;
#pragma unroll
            for (int c = 0; c < 16; c++) {
                const uint32_t v = (acc[8 * h + (c >> 1)] >> (16 * (c & 1))) & 0xffffu;
                if (v) atomicAdd(&table[tb * 512 + (row + 16 * h) * 16 + c], v);
            }
        }
    }
    constexpr int kFirstBallotRow = NACC == 16 ? 32 : 16;
    const uint32_t tb = lane >> 4, cell = lane & 15u;
#pragma unroll
    for (int j = kFirstBallotRow; j < 2 * NACC; j++) {
        if (j >= rows) break;
        const uint32_t v = (acc[j >> 1] >> (16 * (j & 1))) & 0xffffu;
        if (v) atomicAdd(&table[tb * 512 + j * 16 + cell], v);
    }
#pragma unroll
    for (int i = 0; i < NACC; i++) acc[i] = 0;
}

// ---------------------------------------------------------------------------
// building blocks of the tally kernel
// ---------------------------------------------------------------------------
// zero the CTA tables and mirror the contig table into shared memory (24 human
// chromosomes take < 1 KB).  Called by every thread of the CTA.
__device__ __forceinline__ void cta_prologue(TallyShared &T, const TallyArgs &A, uint32_t tid, uint32_t nthreads)
{
    for (uint32_t i = tid; i < 2 * 32 * 16; i += nthreads) T.table[i] = 0;
    if (tid < 8) { T.stats[tid] = 0; T.stats_fk[tid] = 0; }
    const bool fits = A.cc_ok != 0u && A.g.n_contigs <= (uint32_t)kCacheContigs && A.names_bytes <= (uint32_t)kCacheNames && A.g.n_contigs > 0;
    if (fits) {
        for (uint32_t i = tid; i < (uint32_t)kCacheSlots; i += nthreads) T.cc.slot[i] = 0xffu;
        for (uint32_t i = tid; i < (uint32_t)(kCacheNames / 4 + 2 * kCacheContigs); i += nthreads) T.cc.names32[i] = 0u;
        if (tid == 0) {                          // word offsets of the padded names
            uint32_t w = 0;
            for (uint32_t i = 0; i < A.g.n_contigs; i++) {
                T.cc.name_w0[i] = (uint16_t)w;
                w += ((A.g.contigs[i].name_len + 3u) >> 2) + 1u;      // + 1: names shorter than 5 bytes are compared on two words
            }
        }
    }
    __syncthreads();
    if (fits && tid < A.g.n_contigs) {
        const DevContig c = A.g.contigs[tid];
        const GlobalAt  nm{ reinterpret_cast<const uint8_t *>(A.g.names) };
        const int       nw = (int)((c.name_len + 3u) >> 2);
        for (int k = 0; k < nw; k++) T.cc.names32[T.cc.name_w0[tid] + k] = field_word(nm, (int)c.name_off, (int)c.name_len, k);
        const uint32_t h = name_hash_words(nm, (int)c.name_off, (int)c.name_len, A.cc_seed);
        T.cc.slot[h & (kCacheSlots - 1)] = (uint8_t)tid;              // distinct slots: the host checked
        T.cc.name_len[tid] = (uint16_t)c.name_len;
        T.cc.base_off[tid] = c.base_off; T.cc.len[tid] = c.len;
    }
    if (tid == 0) { T.cc.n = fits ? A.g.n_contigs : 0u; T.cc.seed = A.cc_seed; }
    __syncthreads();
}
// CTA tables -> global (after a __syncthreads)
template <int MODE>
__device__ __forceinline__ void cta_epilogue(const TallyShared &T, const TallyArgs &A, uint32_t tid, uint32_t nthreads, int rows)
{
    if (MODE != kModeFragkon) {
        for (uint32_t i = tid; i < 2 * 32 * 16; i += nthreads) {
            const uint32_t v = T.table[i];
            const uint32_t tb = i >> 9, row = (i >> 4) & 31u, cell = i & 15u;
            if (v && (int)row < rows) atomicAdd(A.pss_tables + (size_t)tb * rows * 16 + row * 16 + cell, (unsigned long long)v);
        }
    }
    if (tid < kStN && T.stats[tid]) atomicAdd(A.stats + tid, (unsigned long long)T.stats[tid]);
    if (MODE == kModeBoth && tid < kStN && T.stats_fk[tid]) atomicAdd(A.stats_fk + tid, (unsigned long long)T.stats_fk[tid]);
}

// Exact newline listing (a tile in which some 64-byte slot holds two or more newline candidates -- lines shorter than
// 64 bytes, never real SAM -- or a false candidate): every thread walks
// 2 * kIters consecutive chunks, a block scan orders the counts, a second walk
// stores the first kThreads + 1 positions.  Returns the number of newlines.
__device__ __noinline__ uint32_t list_newlines_generic(TallySmem *Sp, int n_valid, uint32_t one)
{
    TallySmem     &S = *Sp;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, full = 0xffffffffu;
    const int      c0 = (int)tid * 2 * kIters;
    uint32_t       sum = 0;
    for (int k = 0; k < 2 * kIters; k++) {
        if (c0 + k >= n_valid) break;
        uint32_t le32, nl32;
        classify32(S.bytes + 32 * (c0 + k), one, le32, nl32);
        sum += (uint32_t)__popc(nl32);
    }
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(full, inc, d);
        if ((int)lane >= d) inc += t;
    }
    __syncthreads();                                  // warp_sum is free again
    if (lane == 31) S.warp_sum[warp] = inc;
    __syncthreads();
    uint32_t base = 0, total = 0;
    for (int w = 0; w < kWarps; w++) {
        const uint32_t v = S.warp_sum[w];
        if (w < (int)warp) base += v;
        total += v;
    }
    uint32_t ord = base + inc - sum;
    for (int k = 0; k < 2 * kIters; k++) {
        if (c0 + k >= n_valid) break;
        uint32_t le32, nl32;
        classify32(S.bytes + 32 * (c0 + k), one, le32, nl32);
        while (nl32) {
            if (ord <= (uint32_t)kThreads) S.nlpos[ord] = (uint32_t)((c0 + k) * 32 + __ffs((int)nl32) - 1);
            nl32 &= nl32 - 1u;
            ord++;
        }
    }
    return total;
}

// One warp-load of records: this lane's record is [start, pe) with its
// terminator at pe (has == false: no record for the lane).  Parses, filters,
// gathers, tallies, counts outcomes.  All 32 lanes of the warp must call it
// together.  text_done() is called by all of them once none reads bytes or le any more.
template <int MODE, int NACC, int ROWS, class TextDone>
__device__ __forceinline__ void process_batch(const TallyArgs &A, TallyShared &T, const uint8_t *bytes, const uint32_t *le,
                                              bool has, int start, int pe, uint64_t goff,
                                              uint32_t lane, uint32_t (&acc)[NACC ? NACC : 1], int &acc_iters, int rows,
                                              uint32_t &st_acc, uint32_t &st_acc_fk, const TextDone &text_done)
{
    const uint32_t full = 0xffffffffu;
    int            code = has ? (int)kNeedSlow : 99;                    // 99 = no record for this lane
    const SmemAt at{ bytes };
    RecView      r;
    r.flag = 0; r.pos = 0; r.mapq = 0; r.tlen = 0;
    r.rname_off = r.cigar_off = r.seq_off = kPrefix; r.rname_len = r.cigar_len = r.seq_len = 0;
    if (code == kNeedSlow) code = split_fast(at, le, start, pe, r);
    if (code == kNeedSlow) {                                            // rare: glibc sscanf rules
        RecView       rs;
        const SmemRel rel{ bytes + start };
        code = scan11(rel, pe - start, rs);
        r = rs;
        r.rname_off += start; r.cigar_off += start; r.seq_off += start;
    }
    // From here on every lane runs the same straight-line code; lanes whose
    // record did not parse (or that have none) carry valid == false.
    const bool valid = (code == kCounted);
    if (!valid) {                     // a failed parse leaves arbitrary offsets behind: park them on safe bytes
        r.flag = 0; r.pos = 0; r.mapq = 0; r.tlen = 0;
        r.rname_off = r.cigar_off = r.seq_off = kPrefix; r.rname_len = r.cigar_len = r.seq_len = 0;
    }
    uint64_t   cb, cl;
    const int  ci = lookup_contig(T.cc, A.g, at, r.rname_off, valid ? r.rname_len : 0, cb, cl);
    PssStreams st;
    int        code_fk = code;                                  // fragkon's outcome in the fused mode
    if (MODE != kModePss) {
        FkHits          h;
        const TallyCfg &F = (MODE == kModeBoth) ? A.cfg_fk : A.cfg;
        const int       rc = fk_record(at, r, valid, ci, cb, cl, A.g, F, h);
        if (valid) code_fk = rc;
        if (h.add5) atomicAdd(A.fk_hist + h.idx5, 1ull);
        if (h.add3) atomicAdd(A.fk_hist + (1ull << (2 * F.K)) + h.idx3, 1ull);
    }
    if (MODE != kModeFragkon && NACC == 0) {                     // -r beyond the ballot tally: straight to the global tables
        if (valid)
            code = pss_record_wide(at, r, ci, cb, cl, A.g, A.cfg, [&](int tb, int row, int cell) {
                atomicAdd(A.pss_tables + ((size_t)tb * rows + row) * 16 + cell, 1ull);
            });
    } else if (MODE != kModeFragkon) {
        const int rc = pss_record<SmemAt, (ROWS ? ROWS - 2 : -1)>(at, r, valid, ci, cb, cl, A.g, A.cfg, st);
        if (valid) code = rc;
    } else {
        code = code_fk;
    }
    if (code != 99) log_outcome(A, goff, code);
    __syncwarp();
    text_done();
    if (MODE != kModeFragkon && NACC > 0) {
        tally_rows<NACC, ROWS>(st, acc, rows, lane, A.one);
        if (++acc_iters >= kFlushEvery) { flush_acc<NACC>(acc, rows, lane, T.table); acc_iters = 0; }
    }
    // outcome counters: lane k (< kStN) keeps counter k of this warp in a register (stats[] order: lines, counted,
    // no contig, filtered, parse failure, undefined); they reach shared memory once, at the end of the kernel
    {
        const uint32_t m_any = __ballot_sync(full, code != 99);
        const uint32_t m0 = __ballot_sync(full, code == kCounted);
        const uint32_t m1 = __ballot_sync(full, code == kNoContig);
        const uint32_t m2 = __ballot_sync(full, code == kFiltered);
        const uint32_t m3 = __ballot_sync(full, code == kParseFail);
        const uint32_t m4 = __ballot_sync(full, code == kUndefined);
        const uint32_t mine = lane == 0 ? m_any : lane == 1 ? m0 : lane == 2 ? m1 : lane == 3 ? m2 : lane == 4 ? m3 : m4;
        st_acc += (uint32_t)__popc(mine);
        if (MODE == kModeBoth) {
            const uint32_t f0 = __ballot_sync(full, code_fk == kCounted);
            const uint32_t f1 = __ballot_sync(full, code_fk == kNoContig);
            const uint32_t f2 = __ballot_sync(full, code_fk == kFiltered);
            const uint32_t f3 = __ballot_sync(full, code_fk == kParseFail);
            const uint32_t f4 = __ballot_sync(full, code_fk == kUndefined);
            const uint32_t mine_fk = lane == 0 ? m_any : lane == 1 ? f0 : lane == 2 ? f1 : lane == 3 ? f2 : lane == 4 ? f3 : f4;
            st_acc_fk += (uint32_t)__popc(mine_fk);
        }
    }
}

// The copy that stages the tile beginning at pos: its 16-byte aligned source (gsrc) and its size, `want` bytes rounded
// so that kPrefix + size is whole 64-byte slots, at most kStageMax, or the rest of the text if that is less.
__device__ __forceinline__ int stage_size(uint64_t pos, int want, uint64_t len16, uint64_t &gsrc)
{
    gsrc = pos ? ((pos - 1) & ~15ull) : 0;
    want = (want + 16) & ~63; want -= 16;
    if (want > kStageMax) want = kStageMax;
    const uint64_t left = len16 - gsrc;
    return left <= (uint64_t)want ? (int)left : want;
}
__device__ __forceinline__ void stage_copy(TallySmem &S, const uint8_t *src, int nb)
{
    fence_proxy_async();                              // the generic-proxy accesses of the old tile come first
    mbar_expect_tx(&S.bar, (uint32_t)nb);
    bulk_g2s(S.bytes + kPrefix, src, (uint32_t)nb, &S.bar);
}

// ---------------------------------------------------------------------------
// tally kernel.
//
// The text is handed out in ranges (an atomic counter: a CTA that is done
// takes the next one); a CTA owns the records that START in its range and
// walks them in tiles of exactly kThreads records: a tile begins at the byte
// after the last record of the previous one, so in the record phase every lane
// of every warp has a record (a fixed 32 KiB tile left a quarter of the lanes
// idle).  Per tile:
//   stage     one cp.async.bulk (TMA engine) of as many bytes as kThreads
//             records are expected to take (running estimate), on an mbarrier
//             that every warp waits on
//   pass A    a 64-byte slot per thread and step (bank-conflict free quad
//             order): SWAR classification into the "<= 0x20" mask words
//             (stored, the record phase walks them) and newline candidates
//             ("<= 0x20 and bit 1", checked against the byte), ranked on the
//             spot with one ballot and one popcount and kept in a register;
//             two candidates in a slot or a false one: exact listing
//   pass B    scan of the kSegs ballot counts (two shuffles deep), newline
//             positions of ordinals 0..kThreads to shared memory
//   records   one thread per record (process_batch).  When the next tile
//             starts in the same range, each warp arrives at a counter as
//             soon as it has read the last byte of this tile's text, and the
//             last one to arrive issues the next copy while the other warps
//             still tally: the tile needs no block barrier at its end.  Else
//             (first record not found yet, a record longer than the tile, the
//             range ends) a block barrier ends the tile and thread 0 copies.
// ---------------------------------------------------------------------------
// NACC = registers of packed partial sums per lane: 9 cover -r <= 16 (the default is 15), 16 cover -r <= 30;
// 0 = any -r, through pss_record_wide() and global atomics (exact, not tuned).  ROWS = R + 2 as a compile-time
// constant for the default -r 15 (the ballot loop then has no per-row exit test), 0 = taken from the arguments
template <int MODE, int NACC, int ROWS>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) tally_kernel(const __grid_constant__ TallyArgs A)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    TallySmem &S = *reinterpret_cast<TallySmem *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t full = 0xffffffffu;
    const uint32_t lt_mask = (1u << lane) - 1u;

    for (uint32_t i = tid; i < 8; i += kThreads) S.le[kChunks + i] = ~0u;
    if (tid < kPrefix) S.bytes[tid] = 'x';                    // never written by a copy; byte 15 becomes '\n' at offset 0
    if (tid == 0) { S.text_done = 0; mbar_init(&S.bar, 1); fence_mbar_init(); }
    cta_prologue(S.sh, A, tid, kThreads);

    const int      rows = A.cfg.R + 2;
    const uint32_t one = A.one;
    uint32_t       phase = 0;
    uint32_t       acc[NACC ? NACC : 1];
    int            acc_iters = 0;
    uint32_t       st_acc = 0, st_acc_fk = 0;                 // lane k: outcome counter k of this warp
#pragma unroll
    for (int i = 0; i < (NACC ? NACC : 1); i++) acc[i] = 0;
    const uint64_t text_len = A.len_dev ? (uint64_t)__ldg(A.len_dev) : A.len;
    const uint64_t len16 = (text_len + 15) & ~15ull;
    int            est = kStageMax;                           // bytes the next kThreads records are expected to take

    for (;;) {
        // ---- next range ----
        __syncthreads();                                      // everybody is done with ctl (and with the last tile)
        if (tid == 0) S.ctl[0] = atomicAdd(A.range_ctr, 1u);
        __syncthreads();
        const uint64_t range_begin = (uint64_t)S.ctl[0] * A.range_bytes;
        if (range_begin >= text_len) break;
        const uint64_t range_end = (range_begin + A.range_bytes < text_len) ? range_begin + A.range_bytes : text_len;
        uint64_t       pos = range_begin;                     // everything that starts before pos is somebody's business
        bool           want_full = false;
        bool           staged = false;                        // the copy of the tile at pos is already under way

        while (pos < range_end) {
            // ---- stage ----
            uint64_t       gsrc;                                                  // 16-byte aligned source
            const int      nb = stage_size(pos, want_full ? kStageMax : est, len16, gsrc);
            const int64_t  gbase = (int64_t)gsrc - kPrefix;                       // global offset of bytes[0]
            const int      head = (int)((int64_t)pos - 1 - gbase);                // position of the byte before pos: 15..31
            const bool     sees_end = (uint64_t)nb == len16 - gsrc;               // the copy reaches the end of the text
            const bool     is_full = sees_end || nb >= kStageMax;
            const int      data_end = sees_end ? (int)((int64_t)text_len - gbase) : kPrefix + nb;
            if (tid == 0 && !staged) stage_copy(S, A.sam + gsrc, nb);
            mbar_wait(&S.bar, phase);
            phase ^= 1u;

            // bytes before the record start / after the end of the text are neutralised by the thread that scans them
            // (same thread, program order: no barrier).  The end of the buffer terminates the last line.
            const int tail_slot = data_end >> 6;
            const int n_valid = 2 * (sees_end ? tail_slot + 1 : tail_slot);       // chunks that hold text: whole 64-byte slots
            if (tid == 0) {
                S.bytes[kPrefix - 1] = pos == 0 ? '\n' : 'x';
                for (int i = kPrefix; i < head; i++) S.bytes[i] = 'x';
            }
            if (sees_end && tid == (uint32_t)(tail_slot % kThreads)) {            // the thread that scans this slot
                S.bytes[data_end] = '\n';
                for (int i = data_end + 1; i < 64 * (tail_slot + 1); i++) S.bytes[i] = 'x';
            }

            // ---- pass A: classify, rank newlines ----
            constexpr uint32_t kNoNl = 0xfffffu;              // "this slot holds no newline"
            uint32_t pk[kIters];                              // position | rank << 20 of this thread's newline of step it
            uint32_t redo = 0;                                // a slot with two newlines, or a false candidate: exact listing
            const uint32_t r4 = (lane >> 1) & 3u;             // quad swizzle of this lane (see below)
            const uint32_t qo0 = 16u * r4, qo1 = 16u * (1u ^ r4), qo2 = 16u * (2u ^ r4), qo3 = 16u * (3u ^ r4);
            const uint32_t rot16 = 16u * (r4 & 1u), hi_x = r4 >> 1, swz = 16u * r4;
#pragma unroll
            for (int it = 0; it < kIters; it++) {
                pk[it] = kNoNl;
                if (it * 2 * kThreads < n_valid + 8) {                        // block uniform
                    const int      c = 2 * (it * kThreads + (int)tid);           // this thread's two chunks: c, c + 1
                    const uint8_t *src = S.bytes + 32 * c;
                    // the four 16-byte quads of the slot are loaded in the order 0^r, 1^r, 2^r, 3^r, r = (lane / 2) % 4:
                    // the eight lanes of a quarter warp then touch eight different bank groups (in natural order
                    // lanes 64 bytes apart collide four ways).  A mask word in load order is a true mask word with its
                    // halves swapped when r is odd; which of the two chunks it belongs to is r / 2.
                    const uint4    q0 = *reinterpret_cast<const uint4 *>(src + qo0), q1 = *reinterpret_cast<const uint4 *>(src + qo1);
                    const uint4    q2 = *reinterpret_cast<const uint4 *>(src + qo2), q3 = *reinterpret_cast<const uint4 *>(src + qo3);
                    uint32_t le_x, nc_x, le_y, nc_y;
                    classify32_fast(q0, q1, one, le_x, nc_x);
                    classify32_fast(q2, q3, one, le_y, nc_y);
                    le_x = __funnelshift_l(le_x, le_x, rot16);
                    le_y = __funnelshift_l(le_y, le_y, rot16);
                    S.le[c + (int)hi_x] = le_x;
                    S.le[c + 1 - (int)hi_x] = le_y;
                    const bool     has = (nc_x | nc_y) != 0u && c < n_valid;      // slots past the text hold stale bytes
                    const uint32_t b = __ballot_sync(full, has);
                    const uint32_t rank = (uint32_t)__popc(b & lt_mask);
                    const uint32_t x = nc_x ? nc_x : nc_y;
                    // bit index in load order -> byte offset in the slot: the quad index sits in bits 4..5
                    const uint32_t p = (uint32_t)(32 * c) + ((((nc_x ? 0u : 32u) + (uint32_t)__ffs((int)x) - 1u) ^ swz) & 63u);
                    // exactly one candidate in the slot, and it is a '\n'
                    redo |= has ? ((x & (x - 1u)) | (nc_x ? nc_y : 0u) | ((uint32_t)S.bytes[has ? p : 0u] ^ 0x0au)) : 0u;
                    pk[it] = has ? (p + (rank << 20)) : kNoNl;
                    if (lane == 0) S.seg[it * kWarps + (int)warp] = b;
                } else if (lane == 0) {
                    S.seg[it * kWarps + (int)warp] = 0u;
                }
            }
            const int any_multi = __syncthreads_or((int)(redo != 0u));
            if (tid < 8) S.le[n_valid + (int)tid] = ~0u;      // sentinels: every mask walk ends there (read after the next barrier)

            // ---- pass B: newline ordinals -> positions ----
            uint32_t n_nl;
            if (!any_multi) {
                uint32_t v0 = (lane < (uint32_t)kSegs) ? (uint32_t)__popc(S.seg[lane]) : 0u;
                uint32_t v1 = (kSegs > 32 && lane + 32 < (uint32_t)kSegs) ? (uint32_t)__popc(S.seg[lane + 32]) : 0u;
                uint32_t x = v0 | (v1 << 16);
                uint32_t inc = x;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t t = __shfl_up_sync(full, inc, d);
                    if ((int)lane >= d) inc += t;
                }
                const uint32_t tot = __shfl_sync(full, inc, 31);
                const uint32_t ex = inc - x;                   // exclusive, both halves
                n_nl = (tot & 0xffffu) + (tot >> 16);
#pragma unroll
                for (int it = 0; it < kIters; it++) {
                    const int      s = it * kWarps + (int)warp;
                    const uint32_t e = __shfl_sync(full, ex, s & 31);
                    const uint32_t base = (s < 32) ? (e & 0xffffu) : ((tot & 0xffffu) + (e >> 16));
                    const uint32_t v = pk[it];
                    const uint32_t ord = base + (v >> 20);
                    if (v != kNoNl && ord <= (uint32_t)kThreads) S.nlpos[ord] = v & 0xfffffu;
                }
            } else {
                n_nl = list_newlines_generic(&S, n_valid, one);
            }
            __syncthreads();

            const int n_take = (int)n_nl - 1 < kThreads ? (int)n_nl - 1 : kThreads;     // whole records at hand (may be <= 0)

            // ---- where the next tile begins (block-uniform: every thread derives it from the same shared data);
            //      known before the records are looked at, so its first bytes can be on their way to L2 meanwhile ----
            uint64_t next;
            bool     next_full = false;
            if (n_nl == 0) {
                next = (uint64_t)(gbase + data_end);          // no line end in sight yet (only while looking for the first record)
            } else if (n_take <= 0) {
                const uint64_t first = (uint64_t)(gbase + (int)S.nlpos[0] + 1);
                if (first > pos || !is_full) {
                    next = first; next_full = true;           // stage again from the record start, as much as fits
                } else {                                       // a record longer than a tile
                    __syncthreads();
                    if (tid == 0) S.long_end = (first < range_end) ? long_record<MODE>(&A, &S.sh, first, text_len) : first;
                    __syncthreads();
                    next = S.long_end;
                    if (first >= range_end) next = range_end;
                }
            } else {
                const int used = (int)S.nlpos[n_take] - (int)S.nlpos[0];          // bytes of the n_take records
                next = (uint64_t)(gbase + (int)S.nlpos[n_take] + 1);
                const float per = (float)used / (float)n_take;
                int e2 = (int)(per * (float)kThreads * 1.03f) + 768;
                est = e2 > kStageMax ? kStageMax : e2;
                if (tid == 0 && next < range_end) {          // L2 prefetch of the next tile while the records of this one are processed
                    const uint64_t nsrc = (next - 1) & ~15ull;
                    const uint64_t nleft = len16 - nsrc;
                    const uint32_t nbytes = nleft < (uint64_t)est ? (uint32_t)nleft : (uint32_t)(est & ~15);
                    bulk_prefetch_l2(A.sam + nsrc, nbytes);
                }
            }
            // ---- records ----
            const bool early = n_take > 0 && next < range_end;                   // block uniform
            const auto text_done = [&]() {                    // every lane of the warp is past its last read of bytes and le
                if (early && lane == 0 && arrive_count(&S.text_done) % kWarps == kWarps - 1) {
                    uint64_t nsrc;                                                // the last warp: the next tile, as the stage above will see it
                    const int nnb = stage_size(next, est, len16, nsrc);
                    stage_copy(S, A.sam + nsrc, nnb);
                }
            };
            {
                const bool     in = (int)tid < n_take;
                const int      start = in ? (int)S.nlpos[tid] + 1 : kPrefix;
                const int      pe = in ? (int)S.nlpos[tid + 1] : kPrefix;
                const uint64_t goff = (uint64_t)(gbase + start);
                const bool     has = in && start < data_end && goff < range_end;
                if (__any_sync(full, has))
                    process_batch<MODE, NACC, ROWS>(A, S.sh, S.bytes, S.le, has, start, pe, goff, lane, acc, acc_iters, rows, st_acc, st_acc_fk,
                                                    text_done);
                else
                    text_done();
            }

            want_full = next_full;
            pos = next;
            staged = early;
            // the next tile's copy, pass A and pass B overwrite bytes, le and nlpos only once the copy has landed, i.e.
            // after every warp arrived; without an early copy this barrier orders them after the last reads instead
            if (!early) __syncthreads();
        }
    }

    if (MODE != kModeFragkon && NACC > 0) flush_acc<NACC>(acc, rows, lane, S.sh.table);
    if (lane < (uint32_t)kStN) {
        if (st_acc) atomicAdd(&S.sh.stats[lane], st_acc);
        if (MODE == kModeBoth && st_acc_fk) atomicAdd(&S.sh.stats_fk[lane], st_acc_fk);
    }
    __syncthreads();
    cta_epilogue<MODE>(S.sh, A, tid, kThreads, rows);
}

static_assert(sizeof(TallySmem) + 1024 <= 232448 / kCtasPerSm, "the CTAs of the tally kernel must fit one SM");

}  // namespace pssgpu
