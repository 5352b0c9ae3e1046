// pssgpu_internal.h -- what the translation units of libpssgpu.so share: the context, error plumbing, launch timing,
// and the entry into the tally kernels.  Not part of the ABI (include/pssgpu.h is).
#pragma once

#include "../../include/pssgpu.h"

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "pss_record.h"

namespace pssgpu {
constexpr size_t kFeedPiece   = 64ull << 20;     // bytes of SAM text per tally launch when fed from the host
constexpr size_t kCarryCap    = 4ull << 20;      // longest partial line carried between feeds (longer: cut at fgets stretches)
constexpr size_t kStageCap    = kFeedPiece + kCarryCap;

// Owners of CUDA resources.  A release runs on whichever device is current: the code that resets or destroys an owner
// holds a Bind of the context the resource belongs to.
struct DevFree    { void operator()(void *p) const { cudaFree(p); } };
struct HostFree   { void operator()(void *p) const { cudaFreeHost(p); } };
struct EventFree  { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamFree { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
template <class T> using DevPtr  = std::unique_ptr<T, DevFree>;       // device memory
template <class T> using HostPtr = std::unique_ptr<T, HostFree>;      // pinned host memory
using Event  = std::unique_ptr<CUevent_st, EventFree>;
using Stream = std::unique_ptr<CUstream_st, StreamFree>;

// `bytes` of device memory (DevPtr) or pinned host memory (HostPtr) into p.  The old buffer is freed first, so that the
// two never coexist; on failure p is empty.
template <class T, class D>
cudaError_t alloc(std::unique_ptr<T, D> &p, size_t bytes)
{
    static_assert(std::is_same<D, DevFree>::value || std::is_same<D, HostFree>::value, "alloc: device or pinned memory only");
    p.reset();
    void       *raw = nullptr;
    cudaError_t e = std::is_same<D, HostFree>::value ? cudaMallocHost(&raw, bytes) : cudaMalloc(&raw, bytes);
    if (e == cudaSuccess) p.reset(static_cast<T *>(raw));
    return e;
}
inline cudaError_t create(Event &ev, unsigned flags = cudaEventDisableTiming)
{
    ev.reset();
    cudaEvent_t raw = nullptr;
    cudaError_t e = cudaEventCreateWithFlags(&raw, flags);
    if (e == cudaSuccess) ev.reset(raw);
    return e;
}
inline cudaError_t create(Stream &st)            // streams of this library never synchronise with the legacy default stream
{
    st.reset();
    cudaStream_t raw = nullptr;
    cudaError_t  e = cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking);
    if (e == cudaSuccess) st.reset(raw);
    return e;
}

// A genome made resident by pssgpu_genome_upload* or pssgpu_genome_load*: built complete, then moved into its context.
struct Genome {
    DevPtr<uint64_t>  groups;                    // packed bases, 16 per word
    DevPtr<DevContig> contigs;
    DevPtr<char>      names;
    DevPtr<uint32_t>  hash;
    DevPtr<uint64_t>  exc_pos;                   // "other" symbols: sorted positions and their bytes
    DevPtr<uint8_t>   exc_chr;
    uint64_t  n_groups = 0, n_bases = 0, n_contigs = 0;
    uint32_t  names_bytes = 0, hash_mask = 0;
    uint32_t  cc_seed = 0, cc_ok = 0;            // collision-free hash of the contig names for the kernels' shared-memory table
    uint32_t  n_exc = 0;
    bool      exc_overflow = false;

    bool      resident() const { return groups != nullptr; }
    DevGenome view() const;                      // what the kernels read
    uint64_t  hbm_bytes() const;                 // pssgpu_genome_info
};

struct BamIngest;                                // pssgpu_bam.cu
struct BamDelete { void operator()(BamIngest *b) const; };
}  // namespace pssgpu

struct pssgpu_ctx {
    pssgpu::Stream stream;                    // first member, so destroyed last: after every buffer its work may touch
    int          device = -1;
    int          sm_count = 0;
    std::string  err;

    pssgpu::Genome genome;

    // tally
    int       mode = -1;
    pssgpu::TallyCfg  cfg{};
    pssgpu::TallyCfg  cfg_fk{};               // fragkon options of the fused mode
    pssgpu::DevPtr<unsigned long long> d_tables;      // pss: 2*(R+2)*16
    size_t    pss_elems = 0;
    pssgpu::DevPtr<unsigned long long> d_fk;          // fragkon: 2*4^K
    size_t    fk_elems = 0;
    pssgpu::DevPtr<unsigned long long> d_stats;       // 2 x kStN: outcomes, and fragkon's outcomes in the fused mode
    int       tally_grid_pss = 0, tally_grid_fk = 0;
    pssgpu::DevPtr<unsigned int> d_range_ctr;         // work counter of the tally kernel (zeroed before every launch)

    // host feed staging (SAM text pieces; compressed BGZF batches when BAM is fed)
    pssgpu::DevPtr<uint8_t> d_stage[2];
    int       cur = 0;
    size_t    carry_len = 0;
    uint64_t  fed_bytes = 0;                  // bytes handed to pssgpu_feed* since *_begin
    pssgpu::Stream copy_stream;               // H2D staging copies run here, so that the tally of piece i overlaps the copy of piece i + 1
    pssgpu::Event  ev_copied[2], ev_tallied[2];
    std::unique_ptr<pssgpu::BamIngest, pssgpu::BamDelete> bam;     // state of pssgpu_feed_bam (created on first use)

    // timing
    bool      timing = false;
    std::vector<std::pair<pssgpu::Event, pssgpu::Event>> ev;
    std::vector<pssgpu::Event> ev_pool;
    uint64_t  launches = 0, bytes_scanned = 0, h2d_bytes = 0, d2h_bytes = 0;
    double    kernel_ms = 0.0;

    // debug log
    bool      dbg = false;
    pssgpu::DevPtr<uint64_t> d_dbg_off;
    pssgpu::DevPtr<int8_t>   d_dbg_code;
    pssgpu::DevPtr<unsigned long long> d_dbg_n;
    uint64_t  dbg_cap = 0;                    // 0 until the log is allocated
};

namespace pssgpu {

int  fail(pssgpu_ctx *c, int code, const char *fmt, ...);

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return pssgpu::fail(ctx, e_ == cudaErrorMemoryAllocation ? PSSGPU_ENOMEM : PSSGPU_ECUDA, \
                                "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

struct Bind {          // make the context's device current for the duration of a call
    int prev = -1;
    explicit Bind(const pssgpu_ctx *c) { cudaGetDevice(&prev); if (prev != c->device) cudaSetDevice(c->device); else prev = -1; }
    ~Bind() { if (prev >= 0) cudaSetDevice(prev); }
};

// CUDA-event bracket of one kernel launch on ctx->stream (include/pssgpu.h pssgpu_timing)
void time_begin(pssgpu_ctx *c, uint64_t bytes);
void time_end(pssgpu_ctx *c);
void time_collect(pssgpu_ctx *c);       // stream must be idle

// Tally the SAM text [d_sam, d_sam + len) in the context's open mode.  len_dev != nullptr: the real length is read
// from device memory when the kernel starts (`len` is then an upper bound used to size the launch).
int launch_tally_mode(pssgpu_ctx *ctx, const uint8_t *d_sam, size_t len, uint64_t stream_off,
                      const unsigned long long *len_dev = nullptr);

// pssgpu_bam.cu
void bam_reset(pssgpu_ctx *ctx);          // a new tally begins: forget the stream position
int  bam_set_helpers(pssgpu_ctx *ctx, const std::vector<pssgpu_ctx *> &helpers);      // pssgpu_group_feed_bam
void bam_dealing(pssgpu_ctx *ctx, uint64_t *own, std::vector<uint64_t> *per_helper);
int  bam_check(pssgpu_ctx *ctx, bool finishing);   // after a stream sync: PSSGPU_OK or the ingest error the device flagged
                                                   // (finishing: an unfinished block / record left over is an error too)

}  // namespace pssgpu
