// pssgpu_bam.cu -- BGZF / BAM ingest on the device (SURVEY 8f-1): replaces the reference's
// popen("samtools view [-r RG] <bam>") (pss-bam.c:148-162, fragkon.c:84-93).
//
// pssgpu_feed_bam takes the bytes of a BAM file as they are on disk.  The host only frames BGZF blocks (an 18-byte
// header every ~20 KB); everything else runs on the GPU, batch by batch, stream ordered, without a host round trip:
//
//   H2D        the compressed blocks of a batch (<= 256 MiB), double buffered on the copy stream
//   inflate    one warp per BGZF block (pss_inflate.h), persistent warps pulling blocks from a queue; the warp then checks
//              the block's CRC32 (pss_crc32.h), as htslib does
//   prepare    (first batch) BAM header: magic, l_text, the reference dictionary -> device table
//   guess      one warp per block: where does the first record of this block start?  (records ignore block boundaries
//              and carry no sync marks: 32 lanes test 32 offsets at a time for three plausible records in a row), then
//              the chain from there to the end of the block: record starts -> loc[]
//   fix        one warp: verifies every guess against the exit of the chain before it, exactly, starting from the one
//              known entry; a wrong or missing guess is re-walked from the true entry (rare, serial).  Finds the
//              unfinished record at the end of the batch
//   render     one CTA per block: every record -> the SAM line the reference would have parsed (pss_bamrec.h), the RG
//              filter of `samtools view -r`; CTA-level allocation in the text buffer (line order is irrelevant to a tally)
//   carry      the unfinished tail moves in front of the next batch
//   tally      the tally kernel of pss_kernels.cuh over the rendered text; its length comes from device memory
//
// Several GPUs, one file (pssgpu_group_feed_bam): H2D + inflate of a batch may run on another GPU ("helper": the one with
// the fewest batches in flight); the inflated bytes then come over NVLink (cudaMemcpyPeerAsync) and everything from
// `prepare` on runs here, in file order -- the framing state never leaves this GPU.  Streams and events only.
#include "pssgpu_internal.h"

#include <algorithm>
#include <array>
#include <cstdlib>
#include <cstring>

#include "pss_bamrec.h"
#include "pss_crc32.h"
#include "pss_inflate.h"

namespace pssgpu {

constexpr size_t   kBamCarryCap  = 16ull << 20;   // front of the inflated buffer: header / record carried between batches
constexpr size_t   kBamBatchCompDefault = 256ull << 20;   // compressed bytes per batch ($PSSGPU_BAM_BATCH_MB): one warp inflates one
                                                          // ~20 KB block, so a batch must hold several thousand blocks to fill 148 SMs
constexpr uint32_t kBamMaxBlocks = 32768;
constexpr uint32_t kBamLocCap    = 2048;          // record starts per block: 65536 / 38 bytes < 1725, + the carried one
constexpr uint32_t kBamMaxRefs   = 1u << 21;
constexpr uint32_t kBamNone      = 0xffffffffu;
constexpr int      kBamSlots     = 8;             // batches the host may be ahead of the framing GPU when several GPUs inflate
constexpr int      kInfWarps     = 10;            // warps per CTA of the inflate kernel: 7.3 KB of tables each, three CTAs per SM

enum : unsigned {
    kBamOk = 0, kBamErrInflate = 100 /* + pss_inflate.h code */, kBamErrMagic = 200, kBamErrHeaderTooLarge, kBamErrTooManyRefs,
    kBamErrRecord, kBamErrRecordTooLarge, kBamErrTextOverflow, kBamErrTruncated, kBamErrLocOverflow
};

struct BamDesc { uint32_t src_off, c_len, dst_off, isize; };

struct BamState {                     // device resident
    unsigned long long entry;         // offset in ubuf of the first byte not consumed yet
    unsigned long long u_end;         // end of the inflated data of the current batch
    unsigned long long text_len;      // bytes rendered for the current batch (the tally kernel's length)
    unsigned long long n_records, n_dropped;      // rendered / dropped by the RG filter, all batches
    unsigned long long carry_len;
    unsigned long long rewalked;      // blocks whose guess was missing or wrong
    unsigned int hdr_done, error, error_arg, work_ctr;
    int          n_ref;
    unsigned int hdr_len;
};

struct BamIngest {
    // host side framing
    std::vector<uint8_t> carry;       // bytes of an incomplete BGZF block from the previous call
    bool      finished = false;       // `last` seen
    std::string read_group;
    bool      use_rg = false;
    // device, allocated by bam_ensure in two stages: what inflating needs, then what framing needs
    bool      inflate_ready = false, framing_ready = false;
    DevPtr<BamState> d_state;
    DevPtr<uint8_t>  d_ubuf;          // [0, kBamCarryCap) carry, then the inflated batch
    DevPtr<uint8_t>  d_text;
    size_t    text_cap = 0;
    size_t    batch_comp = 0, batch_u = 0;                       // limits of one batch: compressed / inflated bytes
    DevPtr<uint8_t>  d_comp[2];                                  // compressed staging, double buffered
    DevPtr<uint32_t> d_loc;           // kBamMaxBlocks x kBamLocCap record starts (offsets in ubuf)
    DevPtr<uint32_t> d_s, d_e, d_n;                              // per block: guessed start, chain exit, records
    // descriptor slots: two when this context inflates its own batches (slot = the staging buffer, ctx->cur), a ring of
    // kBamSlots when helpers inflate for it -- the host must be able to deal as many batches ahead as the helpers can hold
    DevPtr<BamDesc>  d_desc[kBamSlots];
    HostPtr<BamDesc> h_desc[kBamSlots];
    HostPtr<uint8_t> h_pfx[kBamSlots];                           // a BGZF block that arrived in two feed calls
    Event     ev_ring_copied[kBamSlots], ev_ring_done[kBamSlots];        // ring mode: descriptors copied / batch processed
    int       ring_slot = 0;
    DevPtr<uint8_t>  d_hdr;           // copy of the BAM header (reference names)
    DevPtr<uint32_t> d_ref_off, d_ref_len;
    DevPtr<char>     d_rg;
    DevPtr<uint32_t> d_crc_tab;       // pss_crc32.h tables; null when $PSSGPU_BAM_CRC=0 switches the check off
    bool      check_crc = true;
    int       rg_len = -1;
    int       inflate_grid = 0;
    uint64_t  batches = 0;
    // several GPUs (pssgpu_group_feed_bam): this context frames, renders and tallies; `helpers` inflate batches for it
    std::vector<pssgpu_ctx *> helpers;
    std::vector<Event>        ev_fetched;        // per helper: its inflated batch has been copied over (its buffer is free)
    std::vector<uint64_t>     helper_batches;
    std::vector<std::array<bool, 2>> helper_busy;  // per helper and staging buffer: a batch dealt there has not been inflated yet
    size_t        deal_start = 0;
    cudaEvent_t   desc_reader[kBamSlots] = {};             // a helper's copy that also reads h_desc[i] (its ev_copied)
    DevPtr<unsigned int> d_remote_err;           // error / error_arg of the helper whose batch was fetched last
    uint64_t      dealt = 0, own_batches = 0;
};

// ------------------------------------------------------------------------------------------------------------ kernels
__device__ __forceinline__ void bam_fail(BamState *st, unsigned code, unsigned arg)
{
    if (atomicCAS(&st->error, 0u, code) == 0u) st->error_arg = arg;
}

// an inflate error flagged on the GPU that inflated a batch for this one (pssgpu_group_feed_bam)
__global__ void bam_merge_error_kernel(BamState *st, const unsigned int *remote)
{
    if (remote[0]) bam_fail(st, remote[0], remote[1]);
}

// the register allocation aims at three CTAs per SM (30 warps, 64 registers): the measured best
__global__ void __launch_bounds__(kInfWarps * 32, 3)
bgzf_inflate_kernel(const BamDesc *__restrict__ desc, uint32_t n_blocks, const uint8_t *__restrict__ comp, uint8_t *udata, BamState *st,
                    const uint32_t *__restrict__ crc_tab)
{
    static_assert(sizeof(InflateTables) >= sizeof(uint32_t) * kCrcSmemWords, "the CRC tables borrow the warp's decode tables");
    extern __shared__ __align__(16) unsigned char smem[];
    InflateTables &T = reinterpret_cast<InflateTables *>(smem)[threadIdx.x >> 5];
    const uint32_t lane = threadIdx.x & 31u;
    for (;;) {
        uint32_t b = 0;
        if (lane == 0) b = atomicAdd(&st->work_ctr, 1u);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= n_blocks) break;
        const BamDesc d = desc[b];
        int rc = kInfOk;
        if (d.isize) rc = inflate_block(comp + d.src_off, d.c_len, udata + d.dst_off, d.isize, T);
        if (rc == kInfOk && d.isize && crc_tab) {
            // the CRC32 of the gzip trailer (htslib checks it, so the reference never sees a damaged block): the decode
            // tables are dead now, their shared memory takes the CRC tables; every lane sums its own words (pss_crc32.h)
            uint32_t *ct = reinterpret_cast<uint32_t *>(&T);
            __syncwarp();                                    // the block is written, the decode tables are no longer read
            for (uint32_t i = lane; i < (uint32_t)kCrcSmemWords; i += 32) ct[i] = __ldg(crc_tab + i);
            __syncwarp();
            const uint32_t got = crc32_warp(udata + d.dst_off, d.isize, ct, crc_tab + kCrcXk);
            const uint8_t *tr = comp + d.src_off + d.c_len;
            const uint32_t want = (uint32_t)__ldg(tr) | ((uint32_t)__ldg(tr + 1) << 8) | ((uint32_t)__ldg(tr + 2) << 16) | ((uint32_t)__ldg(tr + 3) << 24);
            if (got != want) rc = kInfCrcMismatch;
        }
        if (rc != kInfOk && lane == 0) bam_fail(st, kBamErrInflate + (unsigned)rc, b);
        __syncwarp();
    }
}

// One warp.  New batch: data end, text cursor; the BAM header if it has not been seen in full yet.
__global__ void __launch_bounds__(32)
bam_prepare_kernel(BamState *st, const uint8_t *ubuf, uint64_t total_u, uint8_t *hdr, uint32_t *ref_off, uint32_t *ref_len)
{
    const uint32_t lane = threadIdx.x;
    const uint64_t u_end = kBamCarryCap + total_u;
    if (lane == 0) { st->u_end = u_end; st->text_len = 0; }
    if (st->hdr_done || st->error) return;
    const uint64_t e0 = st->entry;
    const uint64_t avail = u_end - e0;
    const uint8_t *p = ubuf + e0;
    if (avail < 12) return;
    if (bam_u32(p) != 0x014d4142u) { if (lane == 0) bam_fail(st, kBamErrMagic, bam_u32(p)); return; }      // "BAM\1"
    const uint64_t l_text = bam_u32(p + 4);
    if (12 + l_text > kBamCarryCap) { if (lane == 0) bam_fail(st, kBamErrHeaderTooLarge, (unsigned)l_text); return; }
    if (avail < 12 + l_text) return;
    const uint32_t n_ref = bam_u32(p + 8 + l_text);
    if (n_ref > kBamMaxRefs) { if (lane == 0) bam_fail(st, kBamErrTooManyRefs, n_ref); return; }
    uint64_t q = 12 + l_text;
    for (uint32_t i = 0; i < n_ref; i++) {                         // warp uniform walk of the dictionary
        if (q + 4 > avail) return;
        const uint64_t l_name = bam_u32(p + q);
        if (q + 8 + l_name > avail) return;
        if (q + 8 + l_name > kBamCarryCap) { if (lane == 0) bam_fail(st, kBamErrHeaderTooLarge, i); return; }
        if (lane == 0) { ref_off[i] = (uint32_t)(q + 4); ref_len[i] = l_name ? (uint32_t)(l_name - 1) : 0u; }
        q += 8 + l_name;
    }
    for (uint64_t i = lane; i < q; i += 32) hdr[i] = p[i];
    __syncwarp();
    if (lane == 0) { st->n_ref = (int)n_ref; st->hdr_len = (unsigned)q; st->entry = e0 + q; st->hdr_done = 1u; }
}

// chain of records from x while they start before u1; starts go to loc (at most kBamLocCap).  Returns the exit: the
// start of the first record at or after u1 -- or the start of a record that is not complete within [.., end), or
// kBamNone when a record is malformed (which ends a chain that began at a wrong guess; on the true chain it is an
// error the caller reports).
__device__ __forceinline__ uint32_t bam_chain(const uint8_t *ubuf, uint64_t x, uint64_t u1, uint64_t end, uint32_t *loc, uint32_t &n_out,
                                              bool write)
{
    uint32_t n = 0;
    while (x < u1) {
        if (x + 4 > end) break;
        const uint32_t bs = bam_u32(ubuf + x);
        if (bs < kBamFixed || bs > kBamMaxRecord) { n_out = n; return kBamNone; }
        if (x + 4 + bs > end) break;
        if (write && n < kBamLocCap) loc[n] = (uint32_t)x;
        n++;
        x += 4ull + bs;
    }
    n_out = n;
    return (uint32_t)x;
}

// One warp per BGZF block.
__global__ void __launch_bounds__(128)
bam_guess_kernel(const BamDesc *__restrict__ desc, uint32_t n_blocks, const uint8_t *__restrict__ ubuf, const BamState *st,
                 uint32_t *__restrict__ loc, uint32_t *__restrict__ S, uint32_t *__restrict__ E, uint32_t *__restrict__ N)
{
    const uint32_t b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (b >= n_blocks) return;
    if (!st->hdr_done || st->error) { if (lane == 0) { S[b] = kBamNone; E[b] = 0; N[b] = 0; } return; }
    const uint64_t end = st->u_end, entry = st->entry;
    const int32_t  n_ref = st->n_ref;
    const BamDesc  d = desc[b];
    const uint64_t u0 = kBamCarryCap + d.dst_off, u1 = u0 + d.isize;
    uint64_t s = ~0ull;
    if (entry < u1 && (entry >= u0 || b == 0)) s = entry;          // the known entry lies in this block (or in the carry before block 0)
    else if (entry < u1) {
        for (uint64_t base = u0; base < u1 && s == ~0ull; base += 32) {
            const uint64_t x = base + lane;
            const bool ok = x < u1 && bam_guess_at(ubuf, x, end, n_ref);
            const uint32_t m = __ballot_sync(0xffffffffu, ok);
            if (m) s = base + (uint32_t)__ffs((int)m) - 1u;
        }
    }
    uint32_t n = 0, e = 0;
    if (s != ~0ull) e = bam_chain(ubuf, s, u1, end, loc + (size_t)b * kBamLocCap, n, lane == 0);     // uniform walk, lane 0 writes
    if (lane == 0) { S[b] = s == ~0ull ? kBamNone : (uint32_t)s; E[b] = e; N[b] = n; }
}

// One warp.  Exact verification of the per-block chains, carry of the unfinished tail.
__global__ void __launch_bounds__(32)
bam_fix_kernel(const BamDesc *__restrict__ desc, uint32_t n_blocks, const uint8_t *__restrict__ ubuf, BamState *st,
               uint32_t *__restrict__ loc, uint32_t *__restrict__ S, uint32_t *__restrict__ E, uint32_t *__restrict__ N, int is_last)
{
    const uint32_t lane = threadIdx.x;
    if (st->error) return;
    const uint64_t end = st->u_end;
    uint64_t expected = st->entry;
    unsigned long long rewalked = 0;
    if (st->hdr_done) {
        for (uint32_t base = 0; base < n_blocks; base += 32) {
            const uint32_t b = base + lane;
            const bool     have = b < n_blocks;
            const uint32_t s = have ? S[b] : kBamNone, e = have ? E[b] : 0u;
            const uint32_t u1 = have ? (uint32_t)(kBamCarryCap + desc[b].dst_off + desc[b].isize) : 0u;
            const uint32_t cnt = n_blocks - base < 32u ? n_blocks - base : 32u;
            {   // the usual case in one step: every guess of the group is the exit of the chain before it (lane 0: the
                // known entry) and lies in its own block -- by induction all 32 are true
                const uint32_t pe = __shfl_up_sync(0xffffffffu, e, 1);
                const uint64_t want = lane == 0 ? expected : (uint64_t)pe;
                const bool     good = have && s != kBamNone && e != kBamNone && (uint64_t)s == want && want < (uint64_t)u1;
                if (cnt == 32u && __all_sync(0xffffffffu, good)) { expected = __shfl_sync(0xffffffffu, e, 31); continue; }
            }
            for (uint32_t i = 0; i < cnt; i++) {
                const uint32_t si = __shfl_sync(0xffffffffu, s, (int)i), ei = __shfl_sync(0xffffffffu, e, (int)i);
                const uint32_t u1i = __shfl_sync(0xffffffffu, u1, (int)i);
                if (expected >= u1i) {                        // no record starts in this block (or the chain has ended)
                    if (si != kBamNone && lane == 0) N[base + i] = 0;
                    continue;
                }
                if (si != kBamNone && (uint64_t)si == expected && ei != kBamNone) { expected = ei; continue; }
                // missing or wrong guess: the block is walked again from the true entry
                uint32_t n = 0;
                const uint32_t ee = bam_chain(ubuf, expected, u1i, end, loc + (size_t)(base + i) * kBamLocCap, n, lane == 0);
                rewalked++;
                if (ee == kBamNone) { if (lane == 0) bam_fail(st, kBamErrRecord, base + i); return; }
                if (lane == 0) N[base + i] = n;
                expected = ee;
            }
        }
    }
    // whatever lies between `expected` and the end of the data is an unfinished record (or header): carried over
    const uint64_t carry = end - expected;
    if (lane == 0) {
        st->rewalked += rewalked;
        st->carry_len = carry;
        if (carry > kBamCarryCap) bam_fail(st, kBamErrRecordTooLarge, (unsigned)(carry >> 10));
        else if (is_last && carry) bam_fail(st, kBamErrTruncated, (unsigned)carry);
        st->entry = expected;                              // the carry kernel rebases it
    }
}

// One CTA per BGZF block: records -> SAM lines.  Pass 1, one thread per record: well-formedness, the RG filter, the
// length of the line; a CTA scan gives every line its place and ONE atomic allocates the block's stretch of the text.
// Pass 2, 32 records per warp and round: every lane renders the short head (FLAG .. TLEN) of ONE record into its own
// slot of shared memory -- 32 heads at once instead of one lane at a time -- then the warp goes through the 32 records
// together and stores head, SEQ (4-bit codes -> letters) and QUAL byte by consecutive byte: coalesced stores instead
// of one thread dribbling 240 single bytes.
constexpr int kRenderThreads = 128;
constexpr int kRenderHeadCap = 96;                          // longer heads (long CIGARs / names) are written by their lane directly
constexpr int kRenderHeadStride = 100;                      // 25 words: the 32 slots of a warp start in 32 different banks
// "=ACMGRSVTWYHKDBN"[n] without a (divergent) constant-memory access: the 16 letters sit in four registers
__device__ __forceinline__ uint32_t bam_base_letter(uint32_t n)
{
    const uint32_t lo = __byte_perm(0x4d43413du, 0x56535247u, n & 7u);      // "=ACM" "GRSV"
    const uint32_t hi = __byte_perm(0x48595754u, 0x4e42444bu, n & 7u);      // "TWYH" "KDBN"
    return ((n & 8u) ? hi : lo) & 0xffu;
}
__global__ void __launch_bounds__(kRenderThreads)
bam_render_kernel(const uint8_t *__restrict__ ubuf, BamState *st, const uint32_t *__restrict__ loc, const uint32_t *__restrict__ N,
                  BamRefs refs, const char *__restrict__ rg, int rg_len, uint8_t *__restrict__ text, uint64_t text_cap)
{
    __shared__ uint32_t s_off[kBamLocCap + 1];              // line lengths, then their exclusive prefix sums
    __shared__ uint32_t s_warp[kRenderThreads / 32];
    __shared__ unsigned long long s_base;
    __shared__ uint8_t  s_head[kRenderThreads / 32][32 * kRenderHeadStride];
    const uint32_t b = blockIdx.x, tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (!st->hdr_done || st->error) return;
    const uint32_t n = N[b];
    if (n == 0) return;
    if (n > kBamLocCap) { if (tid == 0) bam_fail(st, kBamErrLocOverflow, b); return; }
    refs.n_ref = st->n_ref;
    const uint32_t *mine = loc + (size_t)b * kBamLocCap;
    // ---- pass 1
    uint32_t dropped = 0;
    for (uint32_t i = tid; i < n; i += kRenderThreads) {
        const uint8_t *r = ubuf + mine[i];
        const BamCore  c = bam_core(r);
        uint32_t       len = 0;
        if (!bam_wellformed(c)) bam_fail(st, kBamErrRecord, b);
        else if (rg_len >= 0 && !bam_has_read_group(r, c, rg, rg_len)) dropped++;
        else {
            BamCountSink cs;
            bam_render_head(r, c, refs, cs);
            len = cs.n + bam_tail_len(c, bam_qual_is_star(r, c));
        }
        s_off[i] = len;
    }
    __syncthreads();
    // exclusive scan of s_off[0 .. n): every thread owns a run of consecutive entries
    const uint32_t per = (n + kRenderThreads - 1) / kRenderThreads, lo = tid * per, hi = lo + per < n ? lo + per : n;
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += s_off[i];
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if ((int)lane >= d) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (uint32_t w = 0; w < kRenderThreads / 32; w++) { const uint32_t v = s_warp[w]; if (w < warp) before += v; total += v; }
    uint32_t run = before + inc - sum;
    for (uint32_t i = lo; i < hi; i++) { const uint32_t v = s_off[i]; s_off[i] = run; run += v; }
    if (tid == 0) { s_off[n] = total; s_base = total ? atomicAdd(&st->text_len, (unsigned long long)total) : 0ull; }
    __syncthreads();
    if (s_base + total > text_cap) { if (tid == 0) bam_fail(st, kBamErrTextOverflow, b); return; }
    // ---- pass 2
    uint8_t *const text_b = text + s_base;
    for (uint32_t i0 = warp * 32u; i0 < n; i0 += kRenderThreads) {
        // this lane's record: the head into the lane's slot, what the cooperative part needs into registers
        const uint32_t i = i0 + lane;
        uint32_t       m_at = 0, m_seq = 0, m_lseq = 0, m_meta = 0;          // meta: head length | QUAL is '*' << 16 | head already stored << 17
        if (i < n) {
            const uint32_t at = s_off[i], len = s_off[i + 1] - at;
            if (len) {                                                  // 0: dropped (RG filter / malformed)
                const uint8_t *r = ubuf + mine[i];
                const BamCore  c = bam_core(r);
                const bool     qs = bam_qual_is_star(r, c);
                const uint32_t head = len - bam_tail_len(c, qs);
                m_at = at; m_lseq = c.l_seq;
                m_seq = (uint32_t)(bam_seq_ptr(r, c) - ubuf);
                m_meta = head | (qs ? 0x10000u : 0u);
                if (head <= (uint32_t)kRenderHeadCap) {
                    BamWriteSink ws{ s_head[warp] + lane * kRenderHeadStride };
                    bam_render_head(r, c, refs, ws);
                } else {
                    BamWriteSink ws{ text_b + at };
                    bam_render_head(r, c, refs, ws);
                    m_meta |= 0x20000u;
                }
                m_meta |= 0x40000u;                                     // a line to write
            }
        }
        __syncwarp();
        const uint32_t cnt = n - i0 < 32u ? n - i0 : 32u;
        for (uint32_t j = 0; j < cnt; j++) {
            const uint32_t meta = __shfl_sync(0xffffffffu, m_meta, (int)j);
            if (!(meta & 0x40000u)) continue;                           // warp uniform
            const uint32_t at = __shfl_sync(0xffffffffu, m_at, (int)j), l_seq = __shfl_sync(0xffffffffu, m_lseq, (int)j);
            const uint8_t *seq = ubuf + __shfl_sync(0xffffffffu, m_seq, (int)j);
            const uint32_t head = meta & 0xffffu;
            const bool     qs = (meta & 0x10000u) != 0u;
            uint8_t       *dst = text_b + at;
            if (!(meta & 0x20000u)) {
                const uint8_t *hs = s_head[warp] + j * kRenderHeadStride;
                for (uint32_t k = lane; k < head; k += 32) dst[k] = hs[k];
            }
            dst += head;
            if (l_seq == 0) {
                if (lane < 4u) dst[lane] = (uint8_t)"*\t*\n"[lane];
                continue;
            }
            // SEQ, tab, QUAL ('I' per base, or '*'), newline
            const uint32_t ql = qs ? 1u : l_seq, tail = l_seq + 1u + ql + 1u;
            for (uint32_t k = lane; k < tail; k += 32) {
                uint32_t v;
                if (k < l_seq) {
                    const uint32_t bb = seq[k >> 1];
                    v = bam_base_letter((k & 1u) ? (bb & 15u) : (bb >> 4));
                } else v = k == l_seq ? (uint32_t)'\t' : k == tail - 1u ? (uint32_t)'\n' : qs ? (uint32_t)'*' : (uint32_t)'I';
                dst[k] = (uint8_t)v;
            }
        }
        __syncwarp();
    }
    // counters: one atomic per warp
#pragma unroll
    for (int d = 16; d; d >>= 1) dropped += __shfl_xor_sync(0xffffffffu, dropped, d);
    if (lane == 0 && dropped) atomicAdd(&st->n_dropped, (unsigned long long)dropped);
    if (tid == 0) atomicAdd(&st->n_records, (unsigned long long)n);
}

// One CTA: the unfinished tail moves to the end of the carry region (an ascending copy to lower addresses: safe when
// source and destination overlap), and the entry follows.
__global__ void __launch_bounds__(256)
bam_carry_kernel(uint8_t *ubuf, BamState *st)
{
    if (st->error) return;
    const uint64_t len = st->carry_len, src = st->entry, dst = kBamCarryCap - len;
    if (src != dst) {
        for (uint64_t off = 0; off < len; off += 256) {
            const uint64_t i = off + threadIdx.x;
            uint8_t v = 0;
            if (i < len) v = ubuf[src + i];
            __syncthreads();
            if (i < len) ubuf[dst + i] = v;
            __syncthreads();
        }
    }
    if (threadIdx.x == 0) st->entry = dst;
}

// ------------------------------------------------------------------------------------------------------------ host side
static const char *bam_error_text(unsigned code)
{
    if (code >= kBamErrInflate && code < kBamErrInflate + 16) {
        static const char *inf[] = { "", "reserved block type", "stored block length check", "invalid code lengths", "invalid literal/length symbol",
                                     "invalid distance", "more data than ISIZE", "compressed data ends early", "less data than ISIZE",
                                     "CRC32 of a BGZF block does not match its data" };
        const unsigned k = code - kBamErrInflate;
        return k < 10 ? inf[k] : "inflate";
    }
    switch (code) {
    case kBamErrMagic: return "not a BAM stream (magic)";
    case kBamErrHeaderTooLarge: return "BAM header larger than 16 MiB";
    case kBamErrTooManyRefs: return "more than 2 M reference sequences";
    case kBamErrRecord: return "malformed alignment record";
    case kBamErrRecordTooLarge: return "alignment record larger than 16 MiB";
    case kBamErrTextOverflow: return "rendered text exceeds its buffer";
    case kBamErrTruncated: return "file ends inside a record or the header";
    case kBamErrLocOverflow: return "more record starts in one BGZF block than the format allows";
    default: return "unknown";
    }
}

void BamDelete::operator()(BamIngest *b) const { delete b; }

void bam_reset(pssgpu_ctx *ctx)
{
    BamIngest *B = ctx->bam.get();
    if (!B) return;
    Bind bind(ctx);
    B->carry.clear();
    B->finished = false;
    B->batches = 0;
    B->dealt = B->own_batches = 0;
    B->deal_start = 0;
    B->ring_slot = 0;
    for (uint64_t &h : B->helper_batches) h = 0;
    for (auto &b : B->helper_busy) b = { false, false };
    if (B->inflate_ready) {
        BamState z;
        memset(&z, 0, sizeof z);
        z.entry = kBamCarryCap;
        cudaMemcpyAsync(B->d_state.get(), &z, sizeof z, cudaMemcpyHostToDevice, ctx->stream.get());
        cudaStreamSynchronize(ctx->stream.get());
    }
    for (pssgpu_ctx *h : B->helpers) bam_reset(h);       // their error flags (a helper need not be a member that *_begin reaches)
}

int bam_check(pssgpu_ctx *ctx, bool finishing)
{
    BamIngest *B = ctx->bam.get();
    if (!B || !B->inflate_ready || B->batches == 0) {
        if (B && finishing && !B->carry.empty())
            return fail(ctx, PSSGPU_EINVAL, "BAM ingest: %zu bytes of an incomplete BGZF block pending (feed with last=1)", B->carry.size());
        return PSSGPU_OK;
    }
    BamState s;
    if (cudaMemcpy(&s, B->d_state.get(), sizeof s, cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, PSSGPU_ECUDA, "BAM ingest: cannot read the device state");
    }
    if (s.error) {
        const int rc = (s.error == kBamErrRecordTooLarge || s.error == kBamErrHeaderTooLarge || s.error == kBamErrTooManyRefs)
                       ? PSSGPU_EUNSUPP : PSSGPU_EINVAL;
        return fail(ctx, rc, "BAM ingest: %s (code %u, at %u)", bam_error_text(s.error), s.error, s.error_arg);
    }
    if (finishing) {
        if (!B->carry.empty())
            return fail(ctx, PSSGPU_EINVAL, "BAM ingest: %zu bytes of an incomplete BGZF block pending (feed with last=1)", B->carry.size());
        if (s.carry_len)
            return fail(ctx, PSSGPU_EINVAL, "BAM ingest: %llu bytes of an unfinished record pending (feed with last=1)", s.carry_len);
    }
    return PSSGPU_OK;
}

namespace {

// inflate_only: the context inflates batches for another one (pssgpu_group_feed_bam) -- the inflated buffer, the
// compressed staging and the inflate tables are all it needs; the framing / rendering buffers (4.8 GB at the default
// batch size) are allocated when the context is first fed a BAM itself
int bam_ensure(pssgpu_ctx *ctx, bool inflate_only = false)
{
    if (!ctx->bam) ctx->bam.reset(new BamIngest());
    BamIngest *B = ctx->bam.get();
    // a stage that failed half way is allocated again from its start: alloc() and create() release what they replace
    if (!B->inflate_ready) {
        size_t mb = kBamBatchCompDefault >> 20;
        if (const char *e = getenv("PSSGPU_BAM_BATCH_MB")) mb = std::min<size_t>(std::max<size_t>(1, strtoull(e, nullptr, 10)), 512);
        B->batch_comp = mb << 20;
        B->batch_u = 6 * B->batch_comp;                        // a batch also closes when its inflated size reaches this
        B->text_cap = 3 * B->batch_u + (64ull << 20);          // lines are ~1.3 x the record bytes; beyond the cap: error, never silence
        CU(alloc(B->d_ubuf, kBamCarryCap + B->batch_u + (1u << 20)));
        for (int i = 0; i < 2; i++) CU(alloc(B->d_comp[i], B->batch_comp + (128u << 10)));
        for (int i = 0; i < kBamSlots; i++) {
            CU(alloc(B->d_desc[i], kBamMaxBlocks * sizeof(BamDesc)));
            CU(alloc(B->h_desc[i], kBamMaxBlocks * sizeof(BamDesc)));
            CU(alloc(B->h_pfx[i], 65536 + 64));
            CU(create(B->ev_ring_copied[i]));
            CU(create(B->ev_ring_done[i]));
        }
        if (const char *e = getenv("PSSGPU_BAM_CRC")) B->check_crc = atoi(e) != 0;
        if (B->check_crc) {
            std::vector<uint32_t> tab(kCrcTableWords);
            crc32_build_tables(tab.data());
            CU(alloc(B->d_crc_tab, tab.size() * sizeof(uint32_t)));
            CU(cudaMemcpy(B->d_crc_tab.get(), tab.data(), tab.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        }
        const size_t smem = (size_t)kInfWarps * sizeof(InflateTables);
        CU(cudaFuncSetAttribute(bgzf_inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bgzf_inflate_kernel, kInfWarps * 32, smem));
        if (occ < 1) return fail(ctx, PSSGPU_ECUDA, "BAM ingest: the inflate kernel does not fit an SM");
        B->inflate_grid = occ * ctx->sm_count;
        CU(cudaMemset(B->d_ubuf.get(), 0, kBamCarryCap));
        BamState z;
        memset(&z, 0, sizeof z);
        z.entry = kBamCarryCap;
        CU(alloc(B->d_state, sizeof(BamState)));
        CU(cudaMemcpy(B->d_state.get(), &z, sizeof z, cudaMemcpyHostToDevice));
        B->inflate_ready = true;
    }
    if (inflate_only || B->framing_ready) return PSSGPU_OK;
    CU(alloc(B->d_text, B->text_cap + 4096));
    CU(alloc(B->d_loc, (size_t)kBamMaxBlocks * kBamLocCap * sizeof(uint32_t)));
    CU(alloc(B->d_s, kBamMaxBlocks * sizeof(uint32_t)));
    CU(alloc(B->d_e, kBamMaxBlocks * sizeof(uint32_t)));
    CU(alloc(B->d_n, kBamMaxBlocks * sizeof(uint32_t)));
    CU(alloc(B->d_hdr, kBamCarryCap + 64));
    CU(alloc(B->d_ref_off, (size_t)kBamMaxRefs * sizeof(uint32_t)));
    CU(alloc(B->d_ref_len, (size_t)kBamMaxRefs * sizeof(uint32_t)));
    CU(alloc(B->d_remote_err, 2 * sizeof(unsigned int)));
    CU(alloc(B->d_rg, 256));
    if (B->use_rg && B->rg_len > 0) CU(cudaMemcpy(B->d_rg.get(), B->read_group.data(), (size_t)B->rg_len, cudaMemcpyHostToDevice));
    B->framing_ready = true;
    return PSSGPU_OK;
}

// One BGZF block at p (n bytes available): its total size, payload offset / length and ISIZE.  Returns 0 when more
// bytes are needed, -1 when p does not start a BGZF block.
int bgzf_frame(const uint8_t *p, size_t n, uint32_t *total, uint32_t *pay_off, uint32_t *pay_len, uint32_t *isize)
{
    if (n < 12) return 0;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return -1;
    const uint32_t xlen = (uint32_t)p[10] | ((uint32_t)p[11] << 8);
    if (n < 12 + (size_t)xlen) return 0;
    uint32_t bsize = 0, at = 12;
    bool     found = false;
    while (at + 4 <= 12 + xlen) {
        const uint32_t slen = (uint32_t)p[at + 2] | ((uint32_t)p[at + 3] << 8);
        if (p[at] == 'B' && p[at + 1] == 'C' && slen == 2 && at + 6 <= 12 + xlen) {
            bsize = (uint32_t)p[at + 4] | ((uint32_t)p[at + 5] << 8);
            found = true;
            break;
        }
        at += 4 + slen;
    }
    if (!found) return -1;
    *total = bsize + 1;
    if (*total < 12 + xlen + 8) return -1;
    if (n < *total) return 0;
    *pay_off = 12 + xlen;
    *pay_len = *total - 12 - xlen - 8;
    *isize = (uint32_t)p[*total - 4] | ((uint32_t)p[*total - 3] << 8) | ((uint32_t)p[*total - 2] << 16) | ((uint32_t)p[*total - 1] << 24);
    if (*isize > 65536u) return -1;
    return 1;
}

// the descriptor slot of the next batch and the events that guard it (see BamIngest)
struct BamSlot { int i; cudaEvent_t copied, done; };
BamSlot bam_slot(pssgpu_ctx *ctx)
{
    BamIngest *B = ctx->bam.get();
    if (B->helpers.empty()) return BamSlot{ ctx->cur, ctx->ev_copied[ctx->cur].get(), ctx->ev_tallied[ctx->cur].get() };
    return BamSlot{ B->ring_slot, B->ev_ring_copied[B->ring_slot].get(), B->ev_ring_done[B->ring_slot].get() };
}

// compressed bytes + block descriptors -> W's staging buffers, inflate on W's stream into W's inflated buffer; `desc` is
// pinned host memory.  W may be the context that frames the batch or a helper on another GPU.
int bam_stage_and_inflate(pssgpu_ctx *W, const uint8_t *pfx, size_t pfx_len, const uint8_t *src, size_t comp_len, const BamDesc *desc,
                          uint32_t n_blocks)
{
    pssgpu_ctx *ctx = W;                                   // (the CU macro reports through `ctx`)
    BamIngest  *B = W->bam.get();
    const int   cur = W->cur;
    // pfx: a block that arrived in two feed calls (pinned copy), in front of the blocks that lie in the caller's buffer
    if (pfx_len) CU(cudaMemcpyAsync(B->d_comp[cur].get(), pfx, pfx_len, cudaMemcpyHostToDevice, W->copy_stream.get()));
    if (comp_len) CU(cudaMemcpyAsync(B->d_comp[cur].get() + pfx_len, src, comp_len, cudaMemcpyHostToDevice, W->copy_stream.get()));
    CU(cudaMemcpyAsync(B->d_desc[cur].get(), desc, n_blocks * sizeof(BamDesc), cudaMemcpyHostToDevice, W->copy_stream.get()));
    W->h2d_bytes += pfx_len + comp_len;
    CU(cudaEventRecord(W->ev_copied[cur].get(), W->copy_stream.get()));
    CU(cudaStreamWaitEvent(W->stream.get(), W->ev_copied[cur].get(), 0));
    cudaStream_t st = W->stream.get();
    CU(cudaMemsetAsync(&B->d_state->work_ctr, 0, sizeof(unsigned int), st));
    const size_t   smem = (size_t)kInfWarps * sizeof(InflateTables);
    const unsigned grid = (unsigned)std::min<uint64_t>((n_blocks + kInfWarps - 1) / kInfWarps, (uint64_t)B->inflate_grid);
    time_begin(W, pfx_len + comp_len);
    bgzf_inflate_kernel<<<grid, kInfWarps * 32, smem, st>>>(B->d_desc[cur].get(), n_blocks, B->d_comp[cur].get(), B->d_ubuf.get() + kBamCarryCap, B->d_state.get(), B->d_crc_tab.get());
    time_end(W);
    CU(cudaGetLastError());
    return PSSGPU_OK;
}

// Submit the blocks framed in h_desc[cur][0 .. n_blocks): compressed bytes pfx[0 .. pfx_len) + [src, src + comp_len) ->
// staging, kernels.  may_deal: with helpers (pssgpu_group_feed_bam) the batch may be inflated on another GPU and fetched
// from there.
int bam_submit(pssgpu_ctx *ctx, const uint8_t *pfx, size_t pfx_len, const uint8_t *src, size_t comp_len, uint32_t n_blocks, uint64_t total_u,
               int is_last, bool may_deal = false)
{
    BamIngest *B = ctx->bam.get();
    const bool    ring = !B->helpers.empty();
    const BamSlot slot = bam_slot(ctx);
    const int     cur = slot.i;
    cudaStream_t st = ctx->stream.get();
    BamState    *S = B->d_state.get();
    int          hi = -1;                                  // helper that inflates this batch
    if (n_blocks && may_deal && !B->helpers.empty()) {
        // the helper with the fewest batches in flight (staged or inflating: at most two, its staging is double buffered);
        // ties go to the first in the list from a rotating start -- the caller lists the other GPUs before the second
        // context on this one, whose inflates share the SMs with the framing / rendering / tallying of every batch
        const size_t nh = B->helpers.size();
        int          best = 3;
        for (size_t k = 0; k < nh; k++) {
            const size_t h = (B->deal_start + k) % nh;
            pssgpu_ctx  *W = B->helpers[h];
            int          fl = 0;
            for (int b = 0; b < 2; b++) {
                if (B->helper_busy[h][b] && cudaEventQuery(W->ev_tallied[b].get()) == cudaSuccess) B->helper_busy[h][b] = false;
                fl += B->helper_busy[h][b] ? 1 : 0;
            }
            cudaGetLastError();                            // (cudaErrorNotReady is an answer, not an error)
            const int cost = 2 * fl + (W->device == ctx->device ? 1 : 0);
            if (cost < best) { best = cost; hi = (int)h; }
        }
        if (hi < 0) hi = (int)(B->deal_start % nh);
        B->deal_start = ((size_t)hi + 1) % nh;
        B->dealt++;
    }
    B->desc_reader[cur] = nullptr;
    if (hi < 0) {
        if (n_blocks) {
            int rc = bam_stage_and_inflate(ctx, pfx, pfx_len, src, comp_len, B->h_desc[cur].get(), n_blocks);
            if (rc != PSSGPU_OK) return rc;
            B->own_batches++;
        } else {
            CU(cudaEventRecord(slot.copied, ctx->copy_stream.get()));
            CU(cudaStreamWaitEvent(st, slot.copied, 0));
        }
    } else {
        pssgpu_ctx *W = B->helpers[hi];
        BamIngest  *Bw = W->bam.get();
        const int   wc = W->cur;
        {
            Bind bind(W);
            // the helper's inflated buffer is free once its previous batch has been fetched
            if (B->helper_batches[hi]) {
                if (cudaStreamWaitEvent(W->stream.get(), B->ev_fetched[hi].get(), 0) != cudaSuccess)
                    return fail(ctx, PSSGPU_ECUDA, "feed_bam: GPU %d cannot wait for GPU %d", W->device, ctx->device);
            }
            int rc = bam_stage_and_inflate(W, pfx, pfx_len, src, comp_len, B->h_desc[cur].get(), n_blocks);
            if (rc == PSSGPU_OK && cudaEventRecord(W->ev_tallied[wc].get(), W->stream.get()) != cudaSuccess) rc = PSSGPU_ECUDA;      // "inflated"
            W->cur ^= 1;
            // its other staging buffer is free once the batch that used it has been inflated
            if (rc == PSSGPU_OK && cudaStreamWaitEvent(W->copy_stream.get(), W->ev_tallied[W->cur].get(), 0) != cudaSuccess) rc = PSSGPU_ECUDA;
            if (rc != PSSGPU_OK) return fail(ctx, rc, "feed_bam: inflate on GPU %d: %s", W->device, pssgpu_last_error(W));
        }
        B->desc_reader[cur] = W->ev_copied[wc].get();
        B->helper_busy[hi][wc] = true;
        B->helper_batches[hi]++;
        // this GPU: the descriptors, then -- once the helper is done -- the inflated bytes and its error flag over NVLink
        CU(cudaMemcpyAsync(B->d_desc[cur].get(), B->h_desc[cur].get(), n_blocks * sizeof(BamDesc), cudaMemcpyHostToDevice, ctx->copy_stream.get()));
        CU(cudaEventRecord(slot.copied, ctx->copy_stream.get()));
        CU(cudaStreamWaitEvent(st, slot.copied, 0));
        CU(cudaStreamWaitEvent(st, W->ev_tallied[wc].get(), 0));
        CU(cudaMemcpyPeerAsync(B->d_ubuf.get() + kBamCarryCap, ctx->device, Bw->d_ubuf.get() + kBamCarryCap, W->device, total_u, st));
        CU(cudaMemcpyPeerAsync(B->d_remote_err.get(), ctx->device, &Bw->d_state->error, W->device, 2 * sizeof(unsigned int), st));
        CU(cudaEventRecord(B->ev_fetched[hi].get(), st));
        bam_merge_error_kernel<<<1, 1, 0, st>>>(S, B->d_remote_err.get());
    }
    bam_prepare_kernel<<<1, 32, 0, st>>>(S, B->d_ubuf.get(), total_u, B->d_hdr.get(), B->d_ref_off.get(), B->d_ref_len.get());
    if (n_blocks) {
        bam_guess_kernel<<<(n_blocks + 3) / 4, 128, 0, st>>>(B->d_desc[cur].get(), n_blocks, B->d_ubuf.get(), S, B->d_loc.get(), B->d_s.get(), B->d_e.get(), B->d_n.get());
    }
    bam_fix_kernel<<<1, 32, 0, st>>>(B->d_desc[cur].get(), n_blocks, B->d_ubuf.get(), S, B->d_loc.get(), B->d_s.get(), B->d_e.get(), B->d_n.get(), is_last);
    if (n_blocks) {
        BamRefs refs;
        refs.blob = B->d_hdr.get(); refs.name_off = B->d_ref_off.get(); refs.name_len = B->d_ref_len.get(); refs.n_ref = 0;
        time_begin(ctx, total_u);
        bam_render_kernel<<<n_blocks, 128, 0, st>>>(B->d_ubuf.get(), S, B->d_loc.get(), B->d_n.get(), refs, B->d_rg.get(), B->use_rg ? B->rg_len : -1,
                                                    B->d_text.get(), B->text_cap);
        time_end(ctx);
    }
    bam_carry_kernel<<<1, 256, 0, st>>>(B->d_ubuf.get(), S);
    CU(cudaGetLastError());
    if (n_blocks) {
        // the text of this batch: at most text_cap bytes, the real length is in the device state
        const size_t bound = std::min<size_t>(B->text_cap, (size_t)(total_u + (1u << 20)) * 3 / 2);
        int rc = launch_tally_mode(ctx, B->d_text.get(), bound, ctx->fed_bytes, &S->text_len);
        if (rc != PSSGPU_OK) return rc;
    }
    CU(cudaEventRecord(slot.done, ctx->stream.get()));
    if (ring) B->ring_slot = (cur + 1) % kBamSlots;
    else ctx->cur ^= 1;
    // the next staging buffer / descriptor slot is free once the batch that used it has been inflated; the simple,
    // sufficient condition: that whole batch is done
    CU(cudaStreamWaitEvent(ctx->copy_stream.get(), bam_slot(ctx).done, 0));
    B->batches++;
    return PSSGPU_OK;
}

int feed_bam_impl(pssgpu_ctx *ctx, const uint8_t *data, size_t len, int last)
{
    BamIngest *B = ctx->bam.get();
    if (B->finished && len) return fail(ctx, PSSGPU_EINVAL, "feed_bam: data after last=1");
    size_t off = 0;
    // a block left incomplete by the previous call is completed in the carry buffer
    while (!B->carry.empty() && off < len) {
        uint32_t total = 0, po = 0, pl = 0, isz = 0;
        int fr = bgzf_frame(B->carry.data(), B->carry.size(), &total, &po, &pl, &isz);
        if (fr < 0) return fail(ctx, PSSGPU_EINVAL, "feed_bam: not a BGZF block (at byte %llu)", (unsigned long long)ctx->fed_bytes);
        if (fr == 1) break;
        // how many more bytes are certainly needed
        size_t need = 1;
        if (B->carry.size() < 12) need = 12 - B->carry.size();
        else {
            const uint32_t xlen = (uint32_t)B->carry[10] | ((uint32_t)B->carry[11] << 8);
            if (B->carry.size() < 12 + (size_t)xlen) need = 12 + xlen - B->carry.size();
            else if (total > B->carry.size()) need = total - B->carry.size();
        }
        const size_t take = std::min(need, len - off);
        B->carry.insert(B->carry.end(), data + off, data + off + take);
        off += take;
    }
    // ... completed now: it becomes the first block of the next batch (through a pinned copy next to the descriptors)
    bool     pfx_pending = false;
    uint32_t pfx_total = 0, pfx_po = 0, pfx_pl = 0, pfx_isz = 0;
    if (!B->carry.empty()) {
        int fr = bgzf_frame(B->carry.data(), B->carry.size(), &pfx_total, &pfx_po, &pfx_pl, &pfx_isz);
        if (fr < 0) return fail(ctx, PSSGPU_EINVAL, "feed_bam: not a BGZF block (at byte %llu)", (unsigned long long)ctx->fed_bytes);
        pfx_pending = fr == 1;
    }
    // whole blocks in place
    while (off < len || pfx_pending) {
        const BamSlot slot = bam_slot(ctx);
        const int     cur = slot.i;
        CU(cudaEventSynchronize(slot.copied));                      // h_desc[cur] / h_pfx[cur] are free again
        if (B->desc_reader[cur]) CU(cudaEventSynchronize(B->desc_reader[cur]));      // ... also on the GPU that inflated that batch
        BamDesc *desc = B->h_desc[cur].get();
        const size_t start = off;
        uint32_t n_blocks = 0, pfx_len = 0;
        uint64_t total_u = 0;
        bool     more = true;
        if (pfx_pending) {
            memcpy(B->h_pfx[cur].get(), B->carry.data(), pfx_total);
            B->carry.clear();
            desc[n_blocks++] = BamDesc{ pfx_po, pfx_pl, 0u, pfx_isz };
            total_u = pfx_isz;
            pfx_len = pfx_total;
            pfx_pending = false;
        }
        while (off < len && n_blocks < kBamMaxBlocks) {
            uint32_t total = 0, po = 0, pl = 0, isz = 0;
            int fr = bgzf_frame(data + off, len - off, &total, &po, &pl, &isz);
            if (fr < 0) return fail(ctx, PSSGPU_EINVAL, "feed_bam: not a BGZF block (at byte %llu)", (unsigned long long)(ctx->fed_bytes + off));
            if (fr == 0) { more = false; break; }
            // the first batch of a stream is a quarter batch: its copy is the one nothing overlaps, the GPU starts sooner
            const size_t comp_cap = B->batches == 0 ? std::max<size_t>(B->batch_comp / 4, 1u << 20) : B->batch_comp;
            if ((off - start) + total > comp_cap || total_u + isz > B->batch_u) break;
            desc[n_blocks++] = BamDesc{ pfx_len + (uint32_t)(off - start) + po, pl, (uint32_t)total_u, isz };
            total_u += isz;
            off += total;
        }
        if (n_blocks) {
            int rc = bam_submit(ctx, B->h_pfx[cur].get(), pfx_len, data + start, off - start, n_blocks, total_u, 0, true);
            if (rc != PSSGPU_OK) return rc;
        }
        if (!more) {                                     // an incomplete block at the end of this call
            B->carry.assign(data + off, data + len);
            off = len;
        }
    }
    ctx->fed_bytes += len;
    if (last) {
        if (!B->carry.empty()) return fail(ctx, PSSGPU_EINVAL, "feed_bam: the stream ends inside a BGZF block (%zu bytes)", B->carry.size());
        // an empty batch with the is_last mark: an unfinished record / header left in the carry is an error
        int rc = bam_submit(ctx, nullptr, 0, nullptr, 0, 0, 0, 1);
        if (rc != PSSGPU_OK) return rc;
        B->finished = true;
    }
    return PSSGPU_OK;
}

}  // namespace

// pssgpu_group_feed_bam: `helpers` (contexts on other GPUs, or -- in tests -- on the same one) inflate batches for ctx
int bam_set_helpers(pssgpu_ctx *ctx, const std::vector<pssgpu_ctx *> &helpers)
{
    {
        Bind bind(ctx);
        int  rc = bam_ensure(ctx);
        if (rc != PSSGPU_OK) return rc;
    }
    BamIngest *B = ctx->bam.get();
    if (B->helpers == helpers) return PSSGPU_OK;
    if (B->batches) return fail(ctx, PSSGPU_EINVAL, "feed_bam: the GPUs of a stream cannot change while it is fed");
    for (pssgpu_ctx *h : helpers) {
        Bind bind(h);
        int  rc = bam_ensure(h, true);
        if (rc != PSSGPU_OK) return fail(ctx, rc, "feed_bam: GPU %d: %s", h->device, pssgpu_last_error(h));
        if (h->bam->batch_comp != B->batch_comp) return fail(ctx, PSSGPU_EINVAL, "feed_bam: GPU %d was set up with another batch size", h->device);
        if (h->device != ctx->device) {                    // peer access both ways where the box has it (otherwise the copy is staged)
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, h->device, ctx->device) == cudaSuccess && can) cudaDeviceEnablePeerAccess(ctx->device, 0);
            cudaGetLastError();
        }
    }
    Bind bind(ctx);
    for (pssgpu_ctx *h : helpers)
        if (h->device != ctx->device) {
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, ctx->device, h->device) == cudaSuccess && can) cudaDeviceEnablePeerAccess(h->device, 0);
            cudaGetLastError();
        }
    B->ev_fetched.clear();
    B->ev_fetched.resize(helpers.size());
    for (Event &e : B->ev_fetched) CU(create(e));
    B->helper_batches.assign(helpers.size(), 0);
    B->helper_busy.assign(helpers.size(), std::array<bool, 2>{ false, false });
    B->deal_start = 0;
    B->helpers = helpers;
    return PSSGPU_OK;
}

// batches inflated on the context's own GPU, and on every helper, since *_begin
void bam_dealing(pssgpu_ctx *ctx, uint64_t *own, std::vector<uint64_t> *per_helper)
{
    BamIngest *B = ctx->bam.get();
    *own = B ? B->own_batches : 0;
    if (B) *per_helper = B->helper_batches; else per_helper->clear();
}

}  // namespace pssgpu

using namespace pssgpu;

extern "C" {

int pssgpu_bam_read_group(pssgpu_ctx *ctx, const char *read_group)
{
    if (!ctx) return PSSGPU_EINVAL;
    Bind bind(ctx);
    int rc = bam_ensure(ctx);
    if (rc != PSSGPU_OK) return rc;
    BamIngest *B = ctx->bam.get();
    CU(cudaStreamSynchronize(ctx->stream.get()));
    if (!read_group) { B->use_rg = false; B->read_group.clear(); B->rg_len = -1; return PSSGPU_OK; }
    const size_t n = strlen(read_group);
    if (n > 255) return fail(ctx, PSSGPU_EUNSUPP, "read group name longer than 255 bytes");
    B->read_group = read_group;
    B->use_rg = true;
    B->rg_len = (int)n;
    if (n) CU(cudaMemcpy(B->d_rg.get(), read_group, n, cudaMemcpyHostToDevice));
    return PSSGPU_OK;
}

int pssgpu_feed_bam(pssgpu_ctx *ctx, const void *bgzf_bytes, size_t len, int last)
{
    if (!ctx || (!bgzf_bytes && len)) return fail(ctx, PSSGPU_EINVAL, "feed_bam: null argument");
    if (ctx->mode < 0) return fail(ctx, PSSGPU_EINVAL, "feed_bam: no tally open (call *_begin first)");
    if (ctx->carry_len) return fail(ctx, PSSGPU_EINVAL, "feed_bam: a partial SAM line from pssgpu_feed is pending");
    Bind bind(ctx);
    int rc = bam_ensure(ctx);
    if (rc == PSSGPU_OK) rc = feed_bam_impl(ctx, (const uint8_t *)bgzf_bytes, len, last);
    // like pssgpu_feed: the caller's bytes have been copied when we return, the kernels may still run
    cudaError_t e = cudaStreamSynchronize(ctx->copy_stream.get());
    for (pssgpu_ctx *h : ctx->bam ? ctx->bam->helpers : std::vector<pssgpu_ctx *>()) {
        const cudaError_t eh = cudaStreamSynchronize(h->copy_stream.get());
        if (e == cudaSuccess) e = eh;
    }
    if (rc != PSSGPU_OK) return rc;
    if (e != cudaSuccess) return fail(ctx, PSSGPU_ECUDA, "feed_bam: %s", cudaGetErrorString(e));
    return PSSGPU_OK;
}

int pssgpu_bam_info(pssgpu_ctx *ctx, pssgpu_bam_stats *out)
{
    if (!ctx || !out) return PSSGPU_EINVAL;
    memset(out, 0, sizeof *out);
    BamIngest *B = ctx->bam.get();
    if (!B || !B->inflate_ready) return PSSGPU_OK;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    BamState s;
    CU(cudaMemcpy(&s, B->d_state.get(), sizeof s, cudaMemcpyDeviceToHost));
    out->records = s.n_records;
    out->dropped_by_read_group = s.n_dropped;
    out->references = s.hdr_done ? (uint64_t)s.n_ref : 0;
    out->batches = B->batches;
    out->blocks_rewalked = s.rewalked;
    return PSSGPU_OK;
}

}  // extern "C"
