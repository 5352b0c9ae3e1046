// pssgpu_internal.h -- what the translation units of libpssgpu.so share: the context, error plumbing, launch timing,
// and the entry into the tally kernels.  Not part of the ABI (include/pssgpu.h is).
#pragma once

#include "../../include/pssgpu.h"

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "pss_record.h"

namespace pssgpu {
constexpr size_t kFeedPiece   = 64ull << 20;     // bytes of SAM text per tally launch when fed from the host
constexpr size_t kCarryCap    = 4ull << 20;      // longest partial line carried between feeds (longer: cut at fgets stretches)
constexpr size_t kStageCap    = kFeedPiece + kCarryCap;
struct BamIngest;                                // pssgpu_bam.cu
}  // namespace pssgpu

struct pssgpu_ctx {
    int          device = -1;
    int          sm_count = 0;
    cudaStream_t stream = nullptr;
    std::string  err;

    // genome
    uint64_t  *d_groups = nullptr;
    uint64_t   n_groups = 0, n_bases = 0, n_contigs = 0, genome_bytes = 0;
    pssgpu::DevContig *d_contigs = nullptr;
    char      *d_names = nullptr;
    uint32_t  *d_hash = nullptr;
    uint32_t   hash_mask = 0;
    uint32_t   names_bytes = 0;
    uint32_t   cc_seed = 0, cc_ok = 0;        // collision-free hash of the contig names for the kernels' shared-memory table
    uint64_t  *d_exc_pos = nullptr;
    uint8_t   *d_exc_chr = nullptr;
    uint32_t   n_exc = 0;
    bool       exc_overflow = false;
    bool       have_genome = false;

    // tally
    int       mode = -1;
    pssgpu::TallyCfg  cfg{};
    pssgpu::TallyCfg  cfg_fk{};               // fragkon options of the fused mode
    unsigned long long *d_tables = nullptr;   // pss: 2*(R+2)*16
    unsigned long long *d_fk = nullptr;       // fragkon: 2*4^K
    size_t    fk_elems = 0;
    unsigned long long *d_stats = nullptr;    // 2 x kStN: outcomes, and fragkon's outcomes in the fused mode
    int       tally_grid_pss = 0, tally_grid_fk = 0;
    unsigned int *d_range_ctr = nullptr;      // work counter of the tally kernel (zeroed before every launch)

    // host feed staging (SAM text pieces; compressed BGZF batches when BAM is fed)
    uint8_t  *d_stage[2] = { nullptr, nullptr };
    int       cur = 0;
    size_t    carry_len = 0;
    uint64_t  fed_bytes = 0;                  // bytes handed to pssgpu_feed* since *_begin
    cudaEvent_t copy_done = nullptr;
    cudaStream_t copy_stream = nullptr;       // H2D staging copies run here, so that the tally of piece i overlaps the copy of piece i + 1
    cudaEvent_t ev_copied[2] = { nullptr, nullptr }, ev_tallied[2] = { nullptr, nullptr };
    pssgpu::BamIngest *bam = nullptr;         // state of pssgpu_feed_bam (created on first use)

    // timing
    bool      timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;
    std::vector<cudaEvent_t> ev_pool;
    uint64_t  launches = 0, bytes_scanned = 0, h2d_bytes = 0, d2h_bytes = 0;
    double    kernel_ms = 0.0;

    // debug log
    bool      dbg = false;
    uint64_t *d_dbg_off = nullptr;
    int8_t   *d_dbg_code = nullptr;
    unsigned long long *d_dbg_n = nullptr;
    uint64_t  dbg_cap = 0;
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
void bam_destroy(pssgpu_ctx *ctx);
int  bam_set_helpers(pssgpu_ctx *ctx, const std::vector<pssgpu_ctx *> &helpers);      // pssgpu_group_feed_bam
void bam_dealing(pssgpu_ctx *ctx, uint64_t *own, std::vector<uint64_t> *per_helper);
int  bam_check(pssgpu_ctx *ctx, bool finishing);   // after a stream sync: PSSGPU_OK or the ingest error the device flagged
                                                   // (finishing: an unfinished block / record left over is an error too)

}  // namespace pssgpu
