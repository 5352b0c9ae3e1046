// pssgpu_group.cu -- several GPUs of one box behind one handle, for the host programs (SURVEY 8e, 8b-3).
//
// One context per GPU in one process.  Reads shard: the caller deals whole lines to the member contexts
// (pssgpu_feed_async); the genome is replicated; every GPU tallies on its own, there is no data-path collective.  The
// only exchange is the sum of the count tables when they are read: one ncclAllReduce(ncclSum, ncclUint64) over
// NVLink / NVSwitch -- 4 352 bytes for pss-bam, 2 x 4^K x 8 for fragkon, 4^k x 8 (128 MiB at k = 12) for the genome-
// sharded spectrum of genome-kmer-count.c:56-58.  NCCL is loaded at run time (libnccl.so.2; the library itself does not
// link it); without it, or with PSSGPU_GROUP_REDUCE=peer, the tables are gathered on the first GPU with peer copies and
// summed there by a small kernel.  Integer sums: the result does not depend on the number of GPUs or on the dealing.
#include "pssgpu_internal.h"

#include <dlfcn.h>
#include <unistd.h>

#include <cstdlib>
#include <cstring>
#include <thread>

using namespace pssgpu;

namespace {

// the few NCCL entry points used, resolved with dlsym (types from nccl.h reduced to what the calls need)
typedef struct ncclComm *ncclComm_t;
struct Nccl {
    void *h = nullptr;
    int (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load()
    {
        if (h) return true;
        for (const char *name : { "libnccl.so.2", "libnccl.so" }) {
            h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) return false;
        CommInitAll = (decltype(CommInitAll))dlsym(h, "ncclCommInitAll");
        CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
        AllReduce = (decltype(AllReduce))dlsym(h, "ncclAllReduce");
        GroupStart = (decltype(GroupStart))dlsym(h, "ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))dlsym(h, "ncclGroupEnd");
        GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
        return CommInitAll && CommDestroy && AllReduce && GroupStart && GroupEnd && GetErrorString;
    }
};
constexpr int kNcclUint64 = 5, kNcclSum = 0;      // nccl.h: ncclUint64, ncclSum

struct CtxDestroy { void operator()(pssgpu_ctx *c) const { pssgpu_destroy(c); } };
using CtxPtr = std::unique_ptr<pssgpu_ctx, CtxDestroy>;

__global__ void add_u64_kernel(unsigned long long *__restrict__ acc, const unsigned long long *__restrict__ x, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc[i] += x[i];
}

}  // namespace

struct pssgpu_group {
    std::vector<CtxPtr>       ctx;
    std::vector<int>          dev;
    std::vector<ncclComm_t>   comm;
    std::vector<DevPtr<unsigned long long>> d_red;  // per GPU: reduction buffer (released under its member's Bind)
    size_t      red_cap = 0;                        // elements
    Nccl        nccl;
    bool        use_nccl = false;
    std::string err;
    size_t      next = 0;                           // round-robin cursor of pssgpu_group_feed
    CtxPtr      bam_self;                           // pssgpu_group_feed_bam: a second context on the first GPU that only inflates
    double      last_reduce_ms = 0.0;
};

namespace {

int gfail(pssgpu_group *g, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (g) g->err = buf;
    return code;
}
int member_fail(pssgpu_group *g, int i, int rc)
{
    return gfail(g, rc, "GPU %d: %s", g->dev[i], pssgpu_last_error(g->ctx[i].get()));
}

int ensure_red(pssgpu_group *g, size_t elems)
{
    if (elems <= g->red_cap) return PSSGPU_OK;
    for (size_t i = 0; i < g->ctx.size(); i++) {
        Bind bind(g->ctx[i].get());
        if (alloc(g->d_red[i], elems * sizeof(unsigned long long)) != cudaSuccess) {
            cudaGetLastError();
            g->red_cap = 0;
            return gfail(g, PSSGPU_ENOMEM, "group: cannot allocate the reduction buffer on GPU %d", g->dev[i]);
        }
    }
    g->red_cap = elems;
    return PSSGPU_OK;
}

// d_red[i][0 .. elems) of every member -> their sum in d_red[0] (and, with NCCL, in every member's buffer)
int reduce_sum(pssgpu_group *g, size_t elems)
{
    const size_t n = g->ctx.size();
    if (n == 1) return PSSGPU_OK;
    Bind bind0(g->ctx[0].get());                    // the timing events and the peer scratch live on the first GPU
    Event e0, e1;
    create(e0, cudaEventDefault);
    create(e1, cudaEventDefault);
    cudaEventRecord(e0.get(), g->ctx[0]->stream.get());
    int rc = PSSGPU_OK;
    if (g->use_nccl) {
        int r = g->nccl.GroupStart();
        for (size_t i = 0; i < n && r == 0; i++) {
            Bind bind(g->ctx[i].get());
            r = g->nccl.AllReduce(g->d_red[i].get(), g->d_red[i].get(), elems, kNcclUint64, kNcclSum, g->comm[i], g->ctx[i]->stream.get());
        }
        const int r2 = g->nccl.GroupEnd();
        if (r == 0) r = r2;
        if (r != 0) rc = gfail(g, PSSGPU_ECUDA, "group: ncclAllReduce: %s", g->nccl.GetErrorString(r));
    } else {
        // peer copies into a scratch area behind the first GPU's own table, added there one by one
        DevPtr<unsigned long long> tmp;
        if (alloc(tmp, elems * sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); rc = gfail(g, PSSGPU_ENOMEM, "group: scratch for the peer reduction"); }
        for (size_t i = 1; i < n && rc == PSSGPU_OK; i++) {
            cudaStreamSynchronize(g->ctx[i]->stream.get());
            cudaError_t e = cudaMemcpyPeerAsync(tmp.get(), g->dev[0], g->d_red[i].get(), g->dev[i], elems * sizeof(unsigned long long), g->ctx[0]->stream.get());
            if (e == cudaSuccess) {
                const unsigned grid = (unsigned)std::min<size_t>((elems + 255) / 256, (size_t)g->ctx[0]->sm_count * 8);
                add_u64_kernel<<<grid, 256, 0, g->ctx[0]->stream.get()>>>(g->d_red[0].get(), tmp.get(), elems);
                e = cudaGetLastError();
            }
            if (e != cudaSuccess) rc = gfail(g, PSSGPU_ECUDA, "group: peer reduction: %s", cudaGetErrorString(e));
        }
        cudaStreamSynchronize(g->ctx[0]->stream.get());      // before tmp is released
    }
    for (size_t i = 0; i < n; i++) {
        Bind bind(g->ctx[i].get());
        if (cudaStreamSynchronize(g->ctx[i]->stream.get()) != cudaSuccess && rc == PSSGPU_OK)
            rc = gfail(g, PSSGPU_ECUDA, "group: reduction failed on GPU %d: %s", g->dev[i], cudaGetErrorString(cudaGetLastError()));
    }
    cudaEventRecord(e1.get(), g->ctx[0]->stream.get());
    cudaEventSynchronize(e1.get());
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e0.get(), e1.get()) == cudaSuccess) g->last_reduce_ms = ms;
    return rc;
}

}  // namespace

namespace {
// tables of every member -> d_red, summed, to the host
template <class Fill>
int gather_sum(pssgpu_group *g, size_t elems, Fill fill, uint64_t *host_out)
{
    int rc = ensure_red(g, elems);
    if (rc != PSSGPU_OK) return rc;
    for (size_t i = 0; i < g->ctx.size(); i++) {
        rc = fill(g->ctx[i].get(), g->d_red[i].get());
        if (rc != PSSGPU_OK) return member_fail(g, (int)i, rc);
    }
    rc = reduce_sum(g, elems);
    if (rc != PSSGPU_OK) return rc;
    Bind bind(g->ctx[0].get());
    if (cudaMemcpy(host_out, g->d_red[0].get(), elems * sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess)
        return gfail(g, PSSGPU_ECUDA, "group: D2H of the summed tables: %s", cudaGetErrorString(cudaGetLastError()));
    return PSSGPU_OK;
}
}  // namespace

extern "C" {

int pssgpu_group_init(const int *devices, int n, pssgpu_group **out)
{
    if (!out) return PSSGPU_EINVAL;
    *out = nullptr;
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess) { cudaGetLastError(); have = 0; }
    std::vector<int> dev;
    if (!devices || n <= 0) { for (int i = 0; i < have; i++) dev.push_back(i); }      // all visible GPUs
    else dev.assign(devices, devices + n);
    if (dev.empty()) return fail(nullptr, PSSGPU_EINVAL, "pssgpu_group_init: no CUDA device");
    // PSSGPU_GROUP_ALLOW_DUP: test switch -- several member contexts on one GPU (a one-GPU box then exercises the
    // dealing and the peer reduction; NCCL refuses two ranks on one device, so it implies the peer path)
    const bool allow_dup = getenv("PSSGPU_GROUP_ALLOW_DUP") != nullptr;
    bool has_dup = false;
    for (size_t i = 0; i < dev.size(); i++)
        for (size_t j = 0; j < i; j++)
            if (dev[i] == dev[j]) {
                if (!allow_dup) return fail(nullptr, PSSGPU_EINVAL, "pssgpu_group_init: device %d listed twice", dev[i]);
                has_dup = true;
            }
    std::unique_ptr<pssgpu_group> g(new pssgpu_group());      // on failure its members are destroyed with it
    g->dev = dev;
    for (int d : dev) {
        pssgpu_ctx *c = nullptr;
        const int rc = pssgpu_init(d, &c);
        if (rc != PSSGPU_OK) return rc;              // pssgpu_last_error(NULL) holds the reason
        g->ctx.emplace_back(c);
    }
    g->d_red.resize(dev.size());
    const char *mode = getenv("PSSGPU_GROUP_REDUCE");
    if (dev.size() > 1 && !has_dup && !(mode && strcmp(mode, "peer") == 0) && g->nccl.load()) {
        g->comm.assign(dev.size(), nullptr);
        // NCCL announces its version on stdout when NCCL_DEBUG asks for it -- stdout is where fragkon and
        // genome-kmer-count print their tables: it goes to stderr for the duration of the initialisation
        fflush(stdout);
        const int saved = dup(1);
        if (saved >= 0) dup2(2, 1);
        const int rc = g->nccl.CommInitAll(g->comm.data(), (int)dev.size(), dev.data());
        fflush(stdout);
        if (saved >= 0) { dup2(saved, 1); close(saved); }
        if (rc == 0) g->use_nccl = true;
        else g->comm.clear();
    }
    if (dev.size() > 1 && !g->use_nccl) {
        // the peer path: the first GPU reads the others' tables
        Bind bind(g->ctx[0].get());
        for (size_t i = 1; i < dev.size(); i++) {
            int can = 0;
            if (dev[i] != dev[0]) cudaDeviceCanAccessPeer(&can, dev[0], dev[i]);
            if (can && cudaDeviceEnablePeerAccess(dev[i], 0) != cudaSuccess) cudaGetLastError();      // (already enabled is fine; without it the copy is staged)
        }
    }
    *out = g.release();
    return PSSGPU_OK;
}

void pssgpu_group_destroy(pssgpu_group *g)
{
    if (!g) return;
    if (g->bam_self) {
        for (CtxPtr &c : g->ctx) { Bind bind(c.get()); cudaStreamSynchronize(c->stream.get()); }      // (they may wait on its events)
        g->bam_self.reset();
    }
    for (size_t i = 0; i < g->ctx.size(); i++) {
        { Bind bind(g->ctx[i].get()); cudaStreamSynchronize(g->ctx[i]->stream.get()); g->d_red[i].reset(); }
        if (g->use_nccl && g->comm[i]) g->nccl.CommDestroy(g->comm[i]);
    }
    delete g;                                        // then the member contexts
}

int         pssgpu_group_size(const pssgpu_group *g) { return g ? (int)g->ctx.size() : 0; }
pssgpu_ctx *pssgpu_group_ctx(pssgpu_group *g, int i) { return (g && i >= 0 && (size_t)i < g->ctx.size()) ? g->ctx[i].get() : nullptr; }
const char *pssgpu_group_last_error(const pssgpu_group *g) { return g ? g->err.c_str() : pssgpu_last_error(nullptr); }
const char *pssgpu_group_reduce_backend(const pssgpu_group *g)
{
    return !g || g->ctx.size() < 2 ? "none (one GPU)" : g->use_nccl ? "nccl" : "peer copies + add kernel";
}
double pssgpu_group_last_reduce_ms(const pssgpu_group *g) { return g ? g->last_reduce_ms : 0.0; }

// Every member packs its own replica; the uploads run on one host thread per GPU (each GPU has its own PCIe link).
int pssgpu_group_genome_upload(pssgpu_group *g, const pssgpu_contig *contigs, uint64_t n_contigs)
{
    if (!g) return PSSGPU_EINVAL;
    std::vector<int> rc(g->ctx.size(), PSSGPU_OK);
    std::vector<std::thread> th;
    for (size_t i = 0; i < g->ctx.size(); i++)
        th.emplace_back([&, i]() { rc[i] = pssgpu_genome_upload(g->ctx[i].get(), contigs, n_contigs); });
    for (auto &t : th) t.join();
    for (size_t i = 0; i < rc.size(); i++)
        if (rc[i] != PSSGPU_OK) return member_fail(g, (int)i, rc[i]);
    return PSSGPU_OK;
}

int pssgpu_group_genome_load_tagged(pssgpu_group *g, const char *path, const pssgpu_genome_tag *expect)
{
    if (!g) return PSSGPU_EINVAL;
    for (size_t i = 0; i < g->ctx.size(); i++) {
        const int rc = pssgpu_genome_load_tagged(g->ctx[i].get(), path, expect);
        if (rc != PSSGPU_OK) return member_fail(g, (int)i, rc);
    }
    return PSSGPU_OK;
}

#define PSS_EACH(call)                                                              \
    do {                                                                            \
        if (!g) return PSSGPU_EINVAL;                                               \
        for (size_t i_ = 0; i_ < g->ctx.size(); i_++) {                             \
            pssgpu_ctx *c = g->ctx[i_].get();                                       \
            const int rc_ = (call);                                                 \
            if (rc_ != PSSGPU_OK) return member_fail(g, (int)i_, rc_);              \
        }                                                                           \
    } while (0)

int pssgpu_group_pss_begin(pssgpu_group *g, const pssgpu_pss_params *p) { PSS_EACH(pssgpu_pss_begin(c, p)); g->next = 0; return PSSGPU_OK; }
int pssgpu_group_fragkon_begin(pssgpu_group *g, const pssgpu_fragkon_params *p) { PSS_EACH(pssgpu_fragkon_begin(c, p)); g->next = 0; return PSSGPU_OK; }
int pssgpu_group_both_begin(pssgpu_group *g, const pssgpu_pss_params *p, const pssgpu_fragkon_params *f)
{
    PSS_EACH(pssgpu_both_begin(c, p, f));
    g->next = 0;
    return PSSGPU_OK;
}
int pssgpu_group_sync(pssgpu_group *g) { PSS_EACH(pssgpu_sync(c)); return PSSGPU_OK; }

// Whole lines only (the last byte of every piece must be '\n' unless `last`): the piece goes to the next member in
// turn.  Returns when the bytes have been copied, like pssgpu_feed; for overlapped copies to several GPUs use
// pssgpu_feed_async on the members (pssgpu_group_ctx), as host/pss_host.c does.
int pssgpu_group_feed(pssgpu_group *g, const char *sam, size_t len, int last)
{
    if (!g || (!sam && len)) return PSSGPU_EINVAL;
    if (len && !last && sam[len - 1] != '\n') return gfail(g, PSSGPU_EINVAL, "group_feed: a piece must end with a newline (lines are dealt whole)");
    const size_t i = g->next++ % g->ctx.size();
    int rc = pssgpu_feed(g->ctx[i].get(), sam, len, 1);          // every piece is a complete text for its member
    if (rc != PSSGPU_OK) return member_fail(g, (int)i, rc);
    return PSSGPU_OK;
}

// A BAM file over the GPUs of the group.  Its byte stream cannot be dealt like text (records run across BGZF blocks and
// carry no sync marks), but the inflate -- five sixths of the ingest -- can: batches of BGZF blocks go to whichever
// GPU has the fewest in flight, every GPU inflates its batches, and the first member fetches the inflated bytes (peer
// copy over NVLink) and frames, renders and tallies them in file order (pssgpu_bam.cu bam_submit).  The first GPU
// inflates too -- through a second context of its own, so that its inflates queue beside, not between, the in-order
// framing of the batches the others deliver; having that work as well, it ends up with fewer batches than they.
int pssgpu_group_feed_bam(pssgpu_group *g, const void *bgzf_bytes, size_t len, int last)
{
    if (!g || (!bgzf_bytes && len)) return PSSGPU_EINVAL;
    pssgpu_ctx *own = g->ctx[0].get();
    std::vector<pssgpu_ctx *> helpers;
    if (g->ctx.size() > 1) {
        if (!g->bam_self) {
            pssgpu_ctx *c = nullptr;
            if (pssgpu_init(g->dev[0], &c) != PSSGPU_OK)
                return gfail(g, PSSGPU_ECUDA, "group_feed_bam: second context on GPU %d: %s", g->dev[0], pssgpu_last_error(nullptr));
            g->bam_self.reset(c);
        }
        for (size_t i = 1; i < g->ctx.size(); i++) helpers.push_back(g->ctx[i].get());
        helpers.push_back(g->bam_self.get());
    }
    int rc = bam_set_helpers(own, helpers);
    if (rc == PSSGPU_OK) rc = pssgpu_feed_bam(own, bgzf_bytes, len, last);
    if (rc != PSSGPU_OK) return member_fail(g, 0, rc);
    return PSSGPU_OK;
}

int pssgpu_group_bam_read_group(pssgpu_group *g, const char *read_group)
{
    if (!g) return PSSGPU_EINVAL;
    const int rc = pssgpu_bam_read_group(g->ctx[0].get(), read_group);
    return rc == PSSGPU_OK ? rc : member_fail(g, 0, rc);
}

// out: what pssgpu_bam_info reports for the member that frames the stream; batches_per_member (may be NULL, one entry
// per member): who inflated how many batches
int pssgpu_group_bam_info(pssgpu_group *g, pssgpu_bam_stats *out, uint64_t *batches_per_member)
{
    if (!g || !out) return PSSGPU_EINVAL;
    const int rc = pssgpu_bam_info(g->ctx[0].get(), out);
    if (rc != PSSGPU_OK) return member_fail(g, 0, rc);
    if (batches_per_member) {
        uint64_t own = 0;
        std::vector<uint64_t> per;
        bam_dealing(g->ctx[0].get(), &own, &per);
        // helpers = members 1 .. n-1, then the second context on the first GPU
        const size_t n = g->ctx.size();
        for (size_t i = 0; i < n; i++) batches_per_member[i] = i == 0 ? own + (per.size() == n ? per[n - 1] : 0) : (i - 1 < per.size() ? per[i - 1] : 0);
    }
    return PSSGPU_OK;
}

int pssgpu_group_pss_finish(pssgpu_group *g, uint64_t *fwd, uint64_t *rev)
{
    if (!g || !fwd || !rev) return PSSGPU_EINVAL;
    const size_t half = (size_t)(g->ctx[0]->cfg.R + 2) * 16;
    std::vector<uint64_t> both(2 * half);
    const int rc = gather_sum(g, 2 * half, [](pssgpu_ctx *c, unsigned long long *d) { return pssgpu_pss_finish_device(c, d); }, both.data());
    if (rc != PSSGPU_OK) return rc;
    memcpy(fwd, both.data(), half * sizeof(uint64_t));
    memcpy(rev, both.data() + half, half * sizeof(uint64_t));
    return PSSGPU_OK;
}

int pssgpu_group_fragkon_finish(pssgpu_group *g, uint64_t *fp, uint64_t *tp)
{
    if (!g || !fp || !tp) return PSSGPU_EINVAL;
    const size_t elems = g->ctx[0]->fk_elems, half = elems / 2;
    if (!elems) return gfail(g, PSSGPU_EINVAL, "group_fragkon_finish: no fragkon tally open");
    std::vector<uint64_t> both(elems);
    const int rc = gather_sum(g, elems, [](pssgpu_ctx *c, unsigned long long *d) { return pssgpu_fragkon_finish_device(c, d); }, both.data());
    if (rc != PSSGPU_OK) return rc;
    memcpy(fp, both.data(), half * sizeof(uint64_t));
    memcpy(tp, both.data() + half, half * sizeof(uint64_t));
    return PSSGPU_OK;
}

int pssgpu_group_get_stats(pssgpu_group *g, pssgpu_stats *out, int fragkon)
{
    if (!g || !out) return PSSGPU_EINVAL;
    memset(out, 0, sizeof *out);
    for (size_t i = 0; i < g->ctx.size(); i++) {
        pssgpu_stats s;
        const int rc = fragkon ? pssgpu_get_fragkon_stats(g->ctx[i].get(), &s) : pssgpu_get_stats(g->ctx[i].get(), &s);
        if (rc != PSSGPU_OK) return member_fail(g, (int)i, rc);
        out->lines += s.lines; out->counted += s.counted; out->no_contig += s.no_contig; out->filtered += s.filtered;
        out->parse_fail += s.parse_fail; out->undefined += s.undefined;
    }
    return PSSGPU_OK;
}

// genome-kmer-count.c:56-58 over the members: GPU i counts slice i of the packed genome (every member holds the whole
// genome; the k-mers are attributed to the slice of their first base), then the 4^k counters are summed.
int pssgpu_group_kmer_spectrum(pssgpu_group *g, int k, uint64_t *counts)
{
    if (!g || !counts) return PSSGPU_EINVAL;
    if (k < 1 || k > kMaxFragK) return gfail(g, PSSGPU_EUNSUPP, "kmer_spectrum: k %d outside [1,%d]", k, kMaxFragK);
    const size_t elems = (size_t)1 << (2 * k);
    int rc = ensure_red(g, elems);
    if (rc != PSSGPU_OK) return rc;
    const int n = (int)g->ctx.size();
    std::vector<int> rcs(n, PSSGPU_OK);
    std::vector<std::thread> th;
    for (int i = 0; i < n; i++)                         // the shard call is synchronous: one host thread per GPU
        th.emplace_back([&, i]() { rcs[i] = pssgpu_kmer_spectrum_shard_device(g->ctx[i].get(), k, i, n, g->d_red[i].get()); });
    for (auto &t : th) t.join();
    for (int i = 0; i < n; i++)
        if (rcs[i] != PSSGPU_OK) return member_fail(g, i, rcs[i]);
    rc = reduce_sum(g, elems);
    if (rc != PSSGPU_OK) return rc;
    Bind bind(g->ctx[0].get());
    if (cudaMemcpy(counts, g->d_red[0].get(), elems * sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess)
        return gfail(g, PSSGPU_ECUDA, "group: D2H of the spectrum: %s", cudaGetErrorString(cudaGetLastError()));
    return PSSGPU_OK;
}

}  // extern "C"
