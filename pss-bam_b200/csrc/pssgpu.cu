// pssgpu.cu -- the C ABI of include/pssgpu.h on top of the sm_100a kernels.
//
// One context = one CUDA device + one stream.  All work of a context is
// stream ordered on that stream: H2D staging copies, pack / tally / spectrum
// kernels and the final D2H of the tables.  There is no CPU implementation of
// any entry point in this library.
#include "pssgpu_internal.h"

#include <unistd.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "pss_kernels.cuh"

using namespace pssgpu;

namespace {
constexpr size_t kPackPiece   = 128ull << 20;    // ASCII bases per pack launch when uploading from the host
constexpr uint64_t kExcCap    = 4ull << 20;      // logged "other" symbols (beyond: -U/-D with such bytes unsupported)
thread_local std::string g_init_error;
}  // namespace

namespace pssgpu {

int fail(pssgpu_ctx *c, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_init_error = buf;
    return code;
}

static Event take_event(pssgpu_ctx *c)
{
    Event e;
    if (!c->ev_pool.empty()) { e = std::move(c->ev_pool.back()); c->ev_pool.pop_back(); return e; }
    create(e, cudaEventDefault);
    return e;
}
void time_begin(pssgpu_ctx *c, uint64_t bytes)
{
    c->launches++;
    c->bytes_scanned += bytes;
    if (!c->timing) return;
    Event a = take_event(c), b = take_event(c);
    cudaEventRecord(a.get(), c->stream.get());
    c->ev.emplace_back(std::move(a), std::move(b));
}
void time_end(pssgpu_ctx *c)
{
    if (!c->timing) return;
    cudaEventRecord(c->ev.back().second.get(), c->stream.get());
}
void time_collect(pssgpu_ctx *c)       // stream must be idle
{
    for (auto &p : c->ev) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.first.get(), p.second.get()) == cudaSuccess) c->kernel_ms += ms;
        c->ev_pool.push_back(std::move(p.first));
        c->ev_pool.push_back(std::move(p.second));
    }
    c->ev.clear();
}

DevGenome Genome::view() const
{
    DevGenome g;
    g.groups = groups.get();   g.n_groups = n_groups;
    g.contigs = contigs.get(); g.n_contigs = (uint32_t)n_contigs;
    g.names = names.get();     g.hash = hash.get(); g.hash_mask = hash_mask;
    g.exc_pos = exc_pos.get(); g.exc_chr = exc_chr.get(); g.n_exc = n_exc;
    return g;
}

uint64_t Genome::hbm_bytes() const
{
    return n_groups * sizeof(uint64_t) + kExcCap * 9 + n_contigs * sizeof(DevContig) + names_bytes + ((uint64_t)hash_mask + 1) * 4;
}

}  // namespace pssgpu

namespace {

// the contig table, the names and their hash table -> g (host tables checked or built by the caller)
cudaError_t put_tables(Genome &g, const DevContig *tab, uint64_t n, const char *names, uint64_t names_bytes, const uint32_t *hash,
                       uint64_t hash_size)
{
    g.n_contigs = n;
    g.names_bytes = (uint32_t)names_bytes;
    g.hash_mask = (uint32_t)(hash_size - 1);
    cudaError_t e = alloc(g.contigs, std::max<size_t>(1, n) * sizeof(DevContig));
    if (e == cudaSuccess) e = alloc(g.names, names_bytes + 16);                  // + slack: names are also read as whole words
    if (e == cudaSuccess) e = alloc(g.hash, hash_size * sizeof(uint32_t));
    if (e == cudaSuccess && n) e = cudaMemcpy(g.contigs.get(), tab, n * sizeof(DevContig), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && names_bytes) e = cudaMemcpy(g.names.get(), names, names_bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(g.hash.get(), hash, hash_size * sizeof(uint32_t), cudaMemcpyHostToDevice);
    return e;
}

int upload_impl(pssgpu_ctx *ctx, const pssgpu_contig *contigs, uint64_t n, bool src_on_device)
{
    if (!ctx || (!contigs && n)) return fail(ctx, PSSGPU_EINVAL, "genome_upload: null argument");
    if (n > 0x7fffffffull) return fail(ctx, PSSGPU_EUNSUPP, "genome_upload: too many contigs");
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    ctx->genome = Genome();          // the old genome goes first: HBM never holds two, and a failed upload leaves none

    // layout + name table
    std::vector<DevContig> tab(n);
    std::string            names;
    uint64_t               cur = kPadBases, total = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (!contigs[i].id || (!contigs[i].seq && contigs[i].len)) return fail(ctx, PSSGPU_EINVAL, "genome_upload: contig %llu has a null field", (unsigned long long)i);
        const size_t nl = strlen(contigs[i].id);
        if (names.size() + nl > 0xfffffff0ull) return fail(ctx, PSSGPU_EUNSUPP, "genome_upload: contig names exceed 4 GiB");
        tab[i].base_off = cur;
        tab[i].len = contigs[i].len;
        tab[i].name_off = (uint32_t)names.size();
        tab[i].name_len = (uint32_t)nl;
        names.append(contigs[i].id, nl);
        cur += ((contigs[i].len + 15) / 16) * 16 + kPadBases;
        total += contigs[i].len;
    }
    {   // find_seq() on duplicate ids depends on qsort/bsearch internals: refuse
        std::vector<uint64_t> order(n);
        for (uint64_t i = 0; i < n; i++) order[i] = i;
        std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return strcmp(contigs[a].id, contigs[b].id) < 0; });
        for (uint64_t i = 1; i < n; i++)
            if (strcmp(contigs[order[i - 1]].id, contigs[order[i]].id) == 0)
                return fail(ctx, PSSGPU_EUNSUPP, "genome_upload: duplicate contig id '%s' (find_seq result would be unspecified)", contigs[order[i]].id);
    }
    const uint64_t n_groups = cur / 16 + 2;       // + slack for the (gi+2) read of a 3-group window
    uint32_t hash_size = 16;
    while (hash_size < 2 * n + 1) hash_size <<= 1;
    std::vector<uint32_t> hash(hash_size, 0);
    for (uint64_t i = 0; i < n; i++) {
        uint32_t h = kNameHashSeed;
        for (uint32_t k = 0; k < tab[i].name_len; k++) h = name_hash_step(h, (uint8_t)names[tab[i].name_off + k]);
        uint32_t slot = h & (hash_size - 1);
        while (hash[slot]) slot = (slot + 1) & (hash_size - 1);
        hash[slot] = (uint32_t)i + 1;
    }

    // seed under which name_hash_words() (pss_kernels.cuh) sends the contig names to distinct slots of the kernels'
    // shared-memory table: one probe per RNAME, no collision chains
    uint32_t cc_seed = 0, cc_ok = 0;
    if (n > 0 && n <= (uint64_t)kCacheContigs && names.size() <= (size_t)kCacheNames) {
        auto host_name_hash = [&](uint64_t i, uint32_t seed) {
            const uint32_t len = tab[i].name_len;
            auto word = [&](uint32_t k) {
                uint32_t w = 0;
                for (uint32_t j = 0; j < 4; j++)
                    if (4 * k + j < len) w |= (uint32_t)(uint8_t)names[tab[i].name_off + 4 * k + j] << (8 * j);
                return w;
            };
            uint32_t       h = seed ^ len;
            const uint32_t nw = (len + 3) >> 2;
            h = (h ^ word(0)) * 0x9E3779B1u;  h ^= h >> 15;
            h = (h ^ word(1)) * 0x9E3779B1u;  h ^= h >> 15;
            for (uint32_t k = 2; k < nw; k++) { h = (h ^ word(k)) * 0x9E3779B1u;  h ^= h >> 15; }
            return h;
        };
        for (uint32_t t = 0; t < 4096 && !cc_ok; t++) {
            const uint32_t seed = kNameHashSeed + t * 0x85EBCA6Bu;
            std::vector<uint8_t> used(kCacheSlots, 0);
            bool clash = false;
            for (uint64_t i = 0; i < n && !clash; i++) {
                uint8_t &u = used[host_name_hash(i, seed) & (kCacheSlots - 1)];
                clash = u != 0;
                u = 1;
            }
            if (!clash) { cc_seed = seed; cc_ok = 1; }
        }
    }

    Genome g;
    DevPtr<uint32_t>           d_flags;
    DevPtr<unsigned long long> d_exc_n;
    DevPtr<uint8_t>            d_piece;
    CU(alloc(g.groups, n_groups * sizeof(uint64_t)));
    CU(cudaMemsetAsync(g.groups.get(), 0xff, n_groups * sizeof(uint64_t), ctx->stream.get()));   // everything "other" until packed
    CU(alloc(g.exc_pos, kExcCap * sizeof(uint64_t)));
    CU(alloc(g.exc_chr, kExcCap));
    CU(alloc(d_flags, sizeof(uint32_t)));
    CU(alloc(d_exc_n, sizeof(unsigned long long)));
    CU(cudaMemsetAsync(d_flags.get(), 0, sizeof(uint32_t), ctx->stream.get()));
    CU(cudaMemsetAsync(d_exc_n.get(), 0, sizeof(unsigned long long), ctx->stream.get()));
    if (!src_on_device) CU(alloc(d_piece, kPackPiece));

    for (uint64_t i = 0; i < n; i++) {
        for (uint64_t off = 0; off < contigs[i].len; off += kPackPiece) {
            const uint64_t nb = std::min<uint64_t>(kPackPiece, contigs[i].len - off);
            PackArgs a;
            if (src_on_device) {
                a.src = reinterpret_cast<const uint8_t *>(contigs[i].seq) + off;
            } else {
                CU(cudaMemcpyAsync(d_piece.get(), contigs[i].seq + off, nb, cudaMemcpyHostToDevice, ctx->stream.get()));
                ctx->h2d_bytes += nb;
                a.src = d_piece.get();
            }
            a.n_bases = nb;
            a.dst = g.groups.get() + (tab[i].base_off + off) / 16;
            a.gbase = tab[i].base_off + off;
            a.exc_pos = g.exc_pos.get(); a.exc_chr = g.exc_chr.get(); a.exc_n = d_exc_n.get(); a.exc_cap = kExcCap;
            a.flags = d_flags.get();
            const uint64_t groups = (nb + 15) / 16;
            const unsigned grid = (unsigned)std::min<uint64_t>((groups + 255) / 256, (uint64_t)ctx->sm_count * 8);
            time_begin(ctx, nb);
            pack_kernel<<<grid, 256, 0, ctx->stream.get()>>>(a);
            time_end(ctx);
            CU(cudaGetLastError());
        }
    }
    uint32_t flags = 0;
    unsigned long long exc_n = 0;
    CU(cudaMemcpyAsync(&flags, d_flags.get(), sizeof flags, cudaMemcpyDeviceToHost, ctx->stream.get()));
    CU(cudaMemcpyAsync(&exc_n, d_exc_n.get(), sizeof exc_n, cudaMemcpyDeviceToHost, ctx->stream.get()));
    CU(cudaStreamSynchronize(ctx->stream.get()));
    time_collect(ctx);
    if (flags & 1u) return fail(ctx, PSSGPU_EUNSUPP, "genome_upload: a contig contains a NUL byte");
    if (exc_n > kExcCap) {
        g.exc_overflow = true;
    } else if (exc_n > 0) {
        std::vector<uint64_t> pos(exc_n);
        std::vector<uint8_t>  chr(exc_n);
        CU(cudaMemcpy(pos.data(), g.exc_pos.get(), exc_n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(chr.data(), g.exc_chr.get(), exc_n, cudaMemcpyDeviceToHost));
        std::vector<uint32_t> order(exc_n);
        for (uint32_t k = 0; k < exc_n; k++) order[k] = k;
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return pos[a] < pos[b]; });
        std::vector<uint64_t> spos(exc_n);
        std::vector<uint8_t>  schr(exc_n);
        for (uint32_t k = 0; k < exc_n; k++) { spos[k] = pos[order[k]]; schr[k] = chr[order[k]]; }
        CU(cudaMemcpy(g.exc_pos.get(), spos.data(), exc_n * sizeof(uint64_t), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(g.exc_chr.get(), schr.data(), exc_n, cudaMemcpyHostToDevice));
        g.n_exc = (uint32_t)exc_n;
    }
    CU(put_tables(g, tab.data(), n, names.data(), names.size(), hash.data(), hash_size));
    g.cc_seed = cc_seed;
    g.cc_ok = cc_ok;
    g.n_groups = n_groups;
    g.n_bases = total;
    ctx->genome = std::move(g);
    return PSSGPU_OK;
}

// bit mask over the 15 named symbols + list of other bytes of a -U / -D string
int ctx_string(pssgpu_ctx *ctx, const char *s, uint32_t *mask, uint32_t *other, char *copy)
{
    static const char named[] = PSSGPU_SYM_CHARS;
    *mask = 0; *other = 0;
    memset(copy, 0, kMaxCtxChars);
    if (!s) return fail(ctx, PSSGPU_EINVAL, "context string is null");
    const size_t n = strlen(s);
    if (n >= (size_t)kMaxCtxChars) return fail(ctx, PSSGPU_EUNSUPP, "context string longer than %d bytes", kMaxCtxChars - 1);
    memcpy(copy, s, n);
    for (size_t i = 0; i < n; i++) {
        const char *p = strchr(named, s[i]);
        if (p && *p) *mask |= 1u << (p - named);
        else *other = 1;      // lower case letters land here too: the genome is upper-cased, they can never match
    }
    return PSSGPU_OK;
}

// The one rule that picks the tally_kernel instantiation for a mode and -r (R is not read in fragkon mode).
// pssgpu_init prepares what it returns for every mode and R; launch_tally_mode launches it.
using TallyKernel = void (*)(TallyArgs);
template <int MODE>
TallyKernel tally_kernel_for_r(int R)
{
    if (R == 15) return tally_kernel<MODE, 9, 17>;              // the default -r
    if (R <= 16) return tally_kernel<MODE, 9, 0>;
    if (R <= kMaxRegion) return tally_kernel<MODE, 16, 0>;
    return tally_kernel<MODE, 0, 0>;                            // any -r: exact, not tuned
}
TallyKernel tally_kernel_for(int mode, int R)
{
    return mode == kModeFragkon ? tally_kernel<kModeFragkon, 9, 0>
         : mode == kModeBoth    ? tally_kernel_for_r<kModeBoth>(R)
                                : tally_kernel_for_r<kModePss>(R);
}

}  // namespace

int pssgpu::launch_tally_mode(pssgpu_ctx *ctx, const uint8_t *d_sam, size_t len, uint64_t stream_off, const unsigned long long *len_dev)
{
    if (len == 0) return PSSGPU_OK;
    TallyArgs a;
    a.sam = d_sam; a.len = len; a.stream_off = stream_off;
    a.len_dev = len_dev;
    a.g = ctx->genome.view();
    a.cfg = ctx->cfg;
    a.cfg_fk = ctx->cfg_fk;
    a.names_bytes = ctx->genome.names_bytes;
    a.cc_seed = ctx->genome.cc_seed;
    a.cc_ok = ctx->genome.cc_ok;
    a.pss_tables = ctx->d_tables.get();
    a.fk_hist = ctx->d_fk.get();
    a.stats = ctx->d_stats.get();
    a.stats_fk = ctx->d_stats.get() + kStN;
    a.dbg_off = ctx->dbg ? ctx->d_dbg_off.get() : nullptr;
    a.dbg_code = ctx->dbg ? ctx->d_dbg_code.get() : nullptr;
    a.dbg_n = ctx->dbg ? ctx->d_dbg_n.get() : nullptr;
    a.dbg_cap = ctx->dbg_cap;
    const int      max_grid = ctx->mode == kModeFragkon ? ctx->tally_grid_fk : ctx->tally_grid_pss;
    // ranges handed out by an atomic counter: about eight per CTA on large inputs, never below 128 KiB
    uint64_t rb = len / ((uint64_t)max_grid * 8u);
    if (const char *e = getenv("PSSGPU_RANGE_KB")) rb = std::max<uint64_t>(1, strtoull(e, nullptr, 10)) << 10;   // developer / test switch
    else rb = std::min<uint64_t>(std::max<uint64_t>(rb, 128u << 10), 1u << 20);
    rb = (rb + 31) & ~31ull;
    const uint64_t n_ranges = (len + rb - 1) / rb;
    a.range_bytes = rb;
    a.range_ctr = ctx->d_range_ctr.get();
    a.one = 1u;
    CU(cudaMemsetAsync(ctx->d_range_ctr.get(), 0, sizeof(unsigned int), ctx->stream.get()));
    time_begin(ctx, len);
    const unsigned grid = (unsigned)std::min<uint64_t>(n_ranges, (uint64_t)max_grid);
    tally_kernel_for(ctx->mode, ctx->cfg.R)<<<grid, kThreads, sizeof(TallySmem), ctx->stream.get()>>>(a);
    time_end(ctx);
    CU(cudaGetLastError());
    return PSSGPU_OK;
}

// ===========================================================================
extern "C" {

int pssgpu_abi_version(void) { return PSSGPU_ABI_VERSION; }

int pssgpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return -1; }
    return n;
}

int pssgpu_init(int device, pssgpu_ctx **out)
{
    pssgpu_ctx *ctx = nullptr;       // CU() reports through g_init_error while ctx is null
    if (!out) return fail(nullptr, PSSGPU_EINVAL, "pssgpu_init: out is null");
    *out = nullptr;
    int n = 0;
    CU(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(nullptr, PSSGPU_EINVAL, "pssgpu_init: device %d of %d", device, n);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, PSSGPU_EUNSUPP, "pssgpu_init: device %d is sm_%d%d; this library holds sm_100a code only",
                    device, prop.major, prop.minor);
    CU(cudaSetDevice(device));
    std::unique_ptr<pssgpu_ctx> c(new pssgpu_ctx());       // on failure released here, with its device current
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    cudaError_t e = create(c->stream);
    if (e == cudaSuccess) e = create(c->copy_stream);
    for (int i = 0; i < 2; i++) {
        if (e == cudaSuccess) e = create(c->ev_copied[i]);
        if (e == cudaSuccess) e = create(c->ev_tallied[i]);
    }
    // every instantiation tally_kernel_for() returns for an accepted -r needs its dynamic shared memory raised above
    // the 48 KB default
    for (int mode : { kModePss, kModeFragkon, kModeBoth }) {
        TallyKernel prev = nullptr;
        for (int R = 0; R <= kMaxRegionWide && e == cudaSuccess; R++) {
            const TallyKernel k = tally_kernel_for(mode, R);
            if (k != prev) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TallySmem));
            prev = k;
        }
    }
    int occ_p = 0, occ_f = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_p, tally_kernel_for(kModePss, kMaxRegion), kThreads, sizeof(TallySmem));
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_f, tally_kernel_for(kModeFragkon, 0), kThreads, sizeof(TallySmem));
    if (e != cudaSuccess || occ_p < 1 || occ_f < 1)
        return fail(nullptr, PSSGPU_ECUDA, "pssgpu_init: %s (occupancy %d/%d)", cudaGetErrorString(e), occ_p, occ_f);
    c->tally_grid_pss = c->sm_count * occ_p;
    c->tally_grid_fk = c->sm_count * occ_f;

    *out = c.release();
    return PSSGPU_OK;
}

void pssgpu_destroy(pssgpu_ctx *ctx)
{
    if (!ctx) return;
    Bind bind(ctx);                   // the context's members are released on its device
    cudaStreamSynchronize(ctx->stream.get());
    delete ctx;
}

const char *pssgpu_last_error(const pssgpu_ctx *ctx) { return ctx ? ctx->err.c_str() : g_init_error.c_str(); }

void *pssgpu_cuda_stream(pssgpu_ctx *ctx) { return ctx ? (void *)ctx->stream.get() : nullptr; }

void *pssgpu_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void pssgpu_host_free(void *p) { if (p) cudaFreeHost(p); }

// ---- genome ---------------------------------------------------------------
int pssgpu_genome_upload(pssgpu_ctx *ctx, const pssgpu_contig *contigs, uint64_t n) { return upload_impl(ctx, contigs, n, false); }
int pssgpu_genome_upload_device(pssgpu_ctx *ctx, const pssgpu_contig *contigs, uint64_t n) { return upload_impl(ctx, contigs, n, true); }

// ---- packed-genome cache ------------------------------------------------------
namespace {
struct CacheHeader {
    char     magic[8];            // "PSSGPUG" + layout version
    uint64_t n_contigs, n_groups, n_bases, names_bytes, n_exc, hash_size;
    uint32_t cc_seed, cc_ok, exc_overflow, pad_bases;
    pssgpu_genome_tag tag;        // what the genome was built from (all zero: untagged)
};
const char kCacheMagic[8] = { 'P', 'S', 'S', 'G', 'P', 'U', 'G', 2 };
constexpr size_t kCachePiece = 64ull << 20;

bool write_dev(FILE *f, const void *d, size_t bytes, std::vector<char> &buf)
{
    for (size_t off = 0; off < bytes; off += kCachePiece) {
        const size_t nb = std::min(kCachePiece, bytes - off);
        if (cudaMemcpy(buf.data(), (const char *)d + off, nb, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
        if (fwrite(buf.data(), 1, nb, f) != nb) return false;
    }
    return true;
}
bool read_dev(FILE *f, void *d, size_t bytes, std::vector<char> &buf)
{
    for (size_t off = 0; off < bytes; off += kCachePiece) {
        const size_t nb = std::min(kCachePiece, bytes - off);
        if (fread(buf.data(), 1, nb, f) != nb) return false;
        if (cudaMemcpy((char *)d + off, buf.data(), nb, cudaMemcpyHostToDevice) != cudaSuccess) return false;
    }
    return true;
}
#define PSS_READ_HOST(f, v, n) ((v).resize(n), (n) == 0 || fread((v).data(), sizeof((v)[0]), (n), (f)) == (size_t)(n))
bool same_tag(const pssgpu_genome_tag &a, const pssgpu_genome_tag &b)
{
    return a.source_size == b.source_size && a.source_mtime_ns == b.source_mtime_ns && a.source_path_hash == b.source_path_hash
        && a.user == b.user;
}

int genome_save_impl(pssgpu_ctx *ctx, const char *path, const pssgpu_genome_tag *tag)
{
    if (!ctx || !path) return fail(ctx, PSSGPU_EINVAL, "genome_save: null argument");
    if (!ctx->genome.resident()) return fail(ctx, PSSGPU_ENOGENOME, "genome_save: no genome resident");
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    // written under a temporary name and renamed: a reader never sees a half-written cache
    const std::string tmp = std::string(path) + ".tmp" + std::to_string((long)getpid());
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) return fail(ctx, PSSGPU_EINVAL, "genome_save: cannot create %s", tmp.c_str());
    CacheHeader h;
    memset(&h, 0, sizeof h);
    memcpy(h.magic, kCacheMagic, 8);
    const Genome &G = ctx->genome;
    h.n_contigs = G.n_contigs; h.n_groups = G.n_groups; h.n_bases = G.n_bases; h.names_bytes = G.names_bytes;
    h.n_exc = G.n_exc; h.hash_size = (uint64_t)G.hash_mask + 1; h.cc_seed = G.cc_seed; h.cc_ok = G.cc_ok;
    h.exc_overflow = G.exc_overflow ? 1u : 0u; h.pad_bases = (uint32_t)kPadBases;
    if (tag) h.tag = *tag;
    std::vector<char> buf(kCachePiece);
    bool ok = fwrite(&h, sizeof h, 1, f) == 1
           && write_dev(f, G.contigs.get(), h.n_contigs * sizeof(DevContig), buf)
           && write_dev(f, G.names.get(), h.names_bytes, buf)
           && write_dev(f, G.hash.get(), h.hash_size * sizeof(uint32_t), buf)
           && write_dev(f, G.exc_pos.get(), h.n_exc * sizeof(uint64_t), buf)
           && write_dev(f, G.exc_chr.get(), h.n_exc, buf)
           && write_dev(f, G.groups.get(), h.n_groups * sizeof(uint64_t), buf);
    ok = (fclose(f) == 0) && ok;
    if (ok && rename(tmp.c_str(), path) != 0) ok = false;
    if (!ok) { remove(tmp.c_str()); return fail(ctx, PSSGPU_EINVAL, "genome_save: writing %s failed", path); }
    ctx->d2h_bytes += h.n_groups * sizeof(uint64_t);
    return PSSGPU_OK;
}

int genome_load_impl(pssgpu_ctx *ctx, const char *path, const pssgpu_genome_tag *expect)
{
    if (!ctx || !path) return fail(ctx, PSSGPU_EINVAL, "genome_load: null argument");
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    ctx->genome = Genome();          // as in upload_impl: the old genome goes first, a failed load leaves none
    FILE *f = fopen(path, "rb");
    if (!f) return fail(ctx, PSSGPU_EINVAL, "genome_load: cannot open %s", path);
    CacheHeader h;
    bool ok = fread(&h, sizeof h, 1, f) == 1 && memcmp(h.magic, kCacheMagic, 8) == 0 && h.pad_bases == (uint32_t)kPadBases;
    uint64_t want = 0;
    if (ok) {
        ok = h.n_contigs <= 0x7fffffffull && h.names_bytes <= 0xfffffff0ull && h.n_exc <= kExcCap && h.n_groups >= 2
          && h.n_groups < (1ull << 40) && h.hash_size >= 16 && (h.hash_size & (h.hash_size - 1)) == 0 && h.hash_size <= (1ull << 32)
          && h.hash_size > 2 * h.n_contigs;
        want = sizeof h + h.n_contigs * sizeof(DevContig) + h.names_bytes + h.hash_size * sizeof(uint32_t) + h.n_exc * 9
             + h.n_groups * sizeof(uint64_t);
        if (ok && (fseek(f, 0, SEEK_END) != 0 || (uint64_t)ftell(f) != want || fseek(f, (long)sizeof h, SEEK_SET) != 0)) ok = false;
    }
    if (!ok) { fclose(f); return fail(ctx, PSSGPU_EINVAL, "genome_load: %s is not a packed genome of this library version", path); }
    if (expect && !same_tag(h.tag, *expect)) {
        fclose(f);
        return fail(ctx, PSSGPU_EINVAL, "genome_load: %s was built from a different source (size / mtime / path tag differs)", path);
    }
    // the small tables are checked on the host before anything is made resident: the kernels index the packed genome
    // with them unchecked
    std::vector<DevContig> tab;
    std::vector<char>      names;
    std::vector<uint32_t>  hash;
    std::vector<uint64_t>  exc_pos;
    std::vector<uint8_t>   exc_chr;
    ok = PSS_READ_HOST(f, tab, h.n_contigs) && PSS_READ_HOST(f, names, h.names_bytes) && PSS_READ_HOST(f, hash, h.hash_size)
      && PSS_READ_HOST(f, exc_pos, h.n_exc) && PSS_READ_HOST(f, exc_chr, h.n_exc);
    const uint64_t total_bases = (h.n_groups - 2) * 16;
    uint64_t sum_len = 0;
    for (uint64_t i = 0; ok && i < h.n_contigs; i++) {
        const DevContig &c = tab[i];
        ok = (c.base_off & 15u) == 0 && c.base_off >= (uint64_t)kPadBases && c.len <= total_bases
          && c.base_off + c.len + (uint64_t)kPadBases <= total_bases + 16
          && (uint64_t)c.name_off + c.name_len <= h.names_bytes;
        if (ok && i > 0) ok = c.base_off >= tab[i - 1].base_off + ((tab[i - 1].len + 15) / 16) * 16 + (uint64_t)kPadBases;
        sum_len += c.len;
    }
    ok = ok && sum_len == h.n_bases;
    uint64_t used = 0;
    for (uint64_t i = 0; ok && i < h.hash_size; i++) { ok = hash[i] <= h.n_contigs; used += hash[i] != 0; }
    ok = ok && used == h.n_contigs;
    for (uint64_t i = 0; ok && i < h.n_exc; i++) ok = exc_pos[i] < total_bases + 32 && (i == 0 || exc_pos[i - 1] < exc_pos[i]);
    if (!ok) { fclose(f); return fail(ctx, PSSGPU_EINVAL, "genome_load: %s is damaged (a table entry is out of range)", path); }

    std::vector<char> buf(kCachePiece);
    Genome g;
    cudaError_t e = put_tables(g, tab.data(), h.n_contigs, names.data(), h.names_bytes, hash.data(), h.hash_size);
    if (e == cudaSuccess) e = alloc(g.exc_pos, kExcCap * sizeof(uint64_t));
    if (e == cudaSuccess) e = alloc(g.exc_chr, kExcCap);
    if (e == cudaSuccess) e = alloc(g.groups, h.n_groups * sizeof(uint64_t));
    if (e == cudaSuccess && h.n_exc) e = cudaMemcpy(g.exc_pos.get(), exc_pos.data(), h.n_exc * sizeof(uint64_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && h.n_exc) e = cudaMemcpy(g.exc_chr.get(), exc_chr.data(), h.n_exc, cudaMemcpyHostToDevice);
    ok = e == cudaSuccess && read_dev(f, g.groups.get(), h.n_groups * sizeof(uint64_t), buf);
    fclose(f);
    if (!ok) {
        cudaGetLastError();
        return fail(ctx, e == cudaErrorMemoryAllocation ? PSSGPU_ENOMEM : PSSGPU_EINVAL, "genome_load: reading %s failed", path);
    }
    g.cc_seed = h.cc_seed; g.cc_ok = h.cc_ok;
    g.n_groups = h.n_groups; g.n_bases = h.n_bases;
    g.n_exc = (uint32_t)h.n_exc; g.exc_overflow = h.exc_overflow != 0;
    ctx->genome = std::move(g);
    ctx->h2d_bytes += h.n_groups * sizeof(uint64_t);
    return PSSGPU_OK;
}
}  // namespace

int pssgpu_genome_save(pssgpu_ctx *ctx, const char *path) { return genome_save_impl(ctx, path, nullptr); }
int pssgpu_genome_load(pssgpu_ctx *ctx, const char *path) { return genome_load_impl(ctx, path, nullptr); }
int pssgpu_genome_save_tagged(pssgpu_ctx *ctx, const char *path, const pssgpu_genome_tag *tag)
{
    if (!tag) return fail(ctx, PSSGPU_EINVAL, "genome_save_tagged: null tag");
    return genome_save_impl(ctx, path, tag);
}
int pssgpu_genome_load_tagged(pssgpu_ctx *ctx, const char *path, const pssgpu_genome_tag *expect)
{
    if (!expect) return fail(ctx, PSSGPU_EINVAL, "genome_load_tagged: null tag");
    return genome_load_impl(ctx, path, expect);
}

int pssgpu_genome_info(const pssgpu_ctx *ctx, uint64_t *n_contigs, uint64_t *n_bases, uint64_t *hbm_bytes)
{
    if (!ctx || !ctx->genome.resident()) return PSSGPU_ENOGENOME;
    if (n_contigs) *n_contigs = ctx->genome.n_contigs;
    if (n_bases) *n_bases = ctx->genome.n_bases;
    if (hbm_bytes) *hbm_bytes = ctx->genome.hbm_bytes();
    return PSSGPU_OK;
}

// ---- pss-bam ----------------------------------------------------------------
void pssgpu_pss_default_params(pssgpu_pss_params *p)
{
    if (!p) return;
    p->region_len = 15;          // pss-bam.c:12
    p->min_len = 0;              // :13
    p->max_len = 250000000UL;    // :14
    p->min_mq = 0;               // :15
    p->up_ctx = "ACGT";          // :16
    p->down_ctx = "ACGT";        // :17
    p->merged_only = 0;          // :18
}

namespace {

int pss_cfg(pssgpu_ctx *ctx, const pssgpu_pss_params *p, TallyCfg &c)
{
    if (p->region_len < 0 || p->region_len > kMaxRegionWide)
        return fail(ctx, PSSGPU_EUNSUPP, "region_len %d outside [0,%d]", p->region_len, kMaxRegionWide);
    c = TallyCfg{};
    c.mode = kModePss;
    c.R = p->region_len;
    c.min_len = p->min_len;
    c.max_len = p->max_len;
    c.min_mq = (uint32_t)p->min_mq;      // `sp->mapq < MIN_MQ` converts MIN_MQ to unsigned (pss-bam.c:409)
    c.merged_only = p->merged_only ? 1u : 0u;
    int rc;
    if ((rc = ctx_string(ctx, p->up_ctx, &c.up_mask, &c.up_other, c.up_ctx)) != PSSGPU_OK) return rc;
    if ((rc = ctx_string(ctx, p->down_ctx, &c.down_mask, &c.down_other, c.down_ctx)) != PSSGPU_OK) return rc;
    if ((c.up_other || c.down_other) && ctx->genome.exc_overflow)
        return fail(ctx, PSSGPU_EUNSUPP, "-U/-D name bytes outside " PSSGPU_SYM_CHARS " and the genome holds more than %llu such bytes",
                    (unsigned long long)kExcCap);
    return PSSGPU_OK;
}

int fk_cfg(pssgpu_ctx *ctx, const pssgpu_fragkon_params *p, TallyCfg &c)
{
    if (p->klen < 1 || p->klen > kMaxFragK) return fail(ctx, PSSGPU_EUNSUPP, "klen %d outside [1,%d]", p->klen, kMaxFragK);
    c = TallyCfg{};
    c.mode = kModeFragkon;
    c.K = p->klen;
    c.min_len = p->min_len;
    c.max_len = p->max_len;
    c.min_mq = (uint32_t)p->min_mq;
    c.merged_only = p->merged_only ? 1u : 0u;
    return PSSGPU_OK;
}

// A zeroed count table of `elems` u64 in buf (of `have` elements), queued on the context's stream.  The buffer is
// replaced only when its size changes; a launch still queued may read the old one, so the stream drains first.
int zero_table(pssgpu_ctx *ctx, DevPtr<unsigned long long> &buf, size_t &have, size_t elems)
{
    if (elems != have) {
        if (buf) CU(cudaStreamSynchronize(ctx->stream.get()));
        have = 0;
        CU(alloc(buf, elems * sizeof(unsigned long long)));
        have = elems;
    }
    CU(cudaMemsetAsync(buf.get(), 0, elems * sizeof(unsigned long long), ctx->stream.get()));
    return PSSGPU_OK;
}

// A new tally: pss (p), fragkon (f) or both from one scan (mode); `fn` names the entry point in messages.  The fused
// mode keeps the pss options in cfg (with cfg.mode == kModeBoth) and the fragkon ones in cfg_fk; fragkon alone keeps
// its options in cfg.
int begin_tally(pssgpu_ctx *ctx, const char *fn, int mode, const pssgpu_pss_params *p, const pssgpu_fragkon_params *f)
{
    const bool pss = mode != kModeFragkon, fk = mode != kModePss;
    if (!ctx || (pss && !p) || (fk && !f)) return fail(ctx, PSSGPU_EINVAL, "%s: null argument", fn);
    if (!ctx->genome.resident()) return fail(ctx, PSSGPU_ENOGENOME, "%s: no genome resident", fn);
    Bind bind(ctx);
    TallyCfg c, cf;
    int rc;
    if (pss && (rc = pss_cfg(ctx, p, c)) != PSSGPU_OK) return rc;
    if (fk && (rc = fk_cfg(ctx, f, cf)) != PSSGPU_OK) return rc;
    // the parameters were accepted: no tally is open until the begin completes (a table it failed to allocate must
    // never be fed)
    ctx->mode = -1;
    // Everything below is queued behind the launches of the previous tally, which may still run, except the BAM
    // ingest bookkeeping bam_reset clears: it describes work on the stream, so a context that ingested BAM drains it.
    // (`cur` stays: copy_stream has already waited for the last tally that read d_stage[cur].)
    if (ctx->bam) CU(cudaStreamSynchronize(ctx->stream.get()));
    if (!ctx->d_stats) CU(alloc(ctx->d_stats, 2 * kStN * sizeof(unsigned long long)));
    if (!ctx->d_range_ctr) CU(alloc(ctx->d_range_ctr, sizeof(unsigned int)));
    CU(cudaMemsetAsync(ctx->d_stats.get(), 0, 2 * kStN * sizeof(unsigned long long), ctx->stream.get()));
    if (ctx->dbg_cap) CU(cudaMemsetAsync(ctx->d_dbg_n.get(), 0, sizeof(unsigned long long), ctx->stream.get()));
    ctx->carry_len = 0;
    ctx->fed_bytes = 0;
    bam_reset(ctx);
    if (pss && (rc = zero_table(ctx, ctx->d_tables, ctx->pss_elems, 2 * (size_t)(c.R + 2) * 16)) != PSSGPU_OK) return rc;
    if (fk && (rc = zero_table(ctx, ctx->d_fk, ctx->fk_elems, 2ull << (2 * cf.K))) != PSSGPU_OK) return rc;
    if (mode == kModeBoth) {
        c.mode = kModeBoth;
        ctx->cfg_fk = cf;
    }
    ctx->cfg = pss ? c : cf;
    ctx->mode = mode;
    return PSSGPU_OK;
}

}  // namespace

int pssgpu_pss_begin(pssgpu_ctx *ctx, const pssgpu_pss_params *p) { return begin_tally(ctx, "pss_begin", kModePss, p, nullptr); }
int pssgpu_fragkon_begin(pssgpu_ctx *ctx, const pssgpu_fragkon_params *p) { return begin_tally(ctx, "fragkon_begin", kModeFragkon, nullptr, p); }
int pssgpu_both_begin(pssgpu_ctx *ctx, const pssgpu_pss_params *p, const pssgpu_fragkon_params *f)
{
    return begin_tally(ctx, "both_begin", kModeBoth, p, f);
}

namespace {
// One piece of the staging buffer `cur` is complete ([0, klen) holds whole lines, or a stretch of one over-long line):
// tally it once its copy has landed, and make the other buffer wait for the tally that last read it.
int stage_launch(pssgpu_ctx *ctx, size_t klen, uint64_t soff)
{
    const int cur = ctx->cur;
    CU(cudaEventRecord(ctx->ev_copied[cur].get(), ctx->copy_stream.get()));
    CU(cudaStreamWaitEvent(ctx->stream.get(), ctx->ev_copied[cur].get(), 0));
    int rc = launch_tally_mode(ctx, ctx->d_stage[cur].get(), klen, soff);
    if (rc != PSSGPU_OK) return rc;
    CU(cudaEventRecord(ctx->ev_tallied[cur].get(), ctx->stream.get()));
    ctx->cur ^= 1;
    CU(cudaStreamWaitEvent(ctx->copy_stream.get(), ctx->ev_tallied[ctx->cur].get(), 0));
    return PSSGPU_OK;
}

int feed_impl(pssgpu_ctx *ctx, const char *sam, size_t len, int last)
{
    for (int s = 0; s < 2; s++)
        if (!ctx->d_stage[s]) CU(alloc(ctx->d_stage[s], kStageCap + 64));
    // Two staging buffers, two streams: the copies queue up on copy_stream, the tallies on the context's stream; a
    // tally waits for its copy (ev_copied), a copy into a buffer waits for the tally that last read it (ev_tallied).
    // The PCIe link then never idles behind a kernel launch.
    size_t off = 0;
    while (off < len) {
        if (ctx->carry_len == kStageCap) {
            // A "line" longer than the staging buffer.  fgets(buf, MAX_LINE_LEN + 1) hands such a line to line2saml in
            // stretches of 200000 bytes (pss-bam.c:761-764), so it may be cut at any multiple of that from its start:
            // the stretches before the cut are tallied now (the kernel's long_record path), the rest stays carried.
            const size_t   cut = (kStageCap / (size_t)kMaxLine) * (size_t)kMaxLine, tail = kStageCap - cut;
            const uint64_t soff = ctx->fed_bytes + off - ctx->carry_len;
            uint8_t       *from = ctx->d_stage[ctx->cur].get();
            int rc = stage_launch(ctx, cut, soff);
            if (rc != PSSGPU_OK) return rc;
            CU(cudaMemcpyAsync(ctx->d_stage[ctx->cur].get(), from + cut, tail, cudaMemcpyDeviceToDevice, ctx->copy_stream.get()));
            ctx->carry_len = tail;
        }
        const size_t room = kStageCap - ctx->carry_len;
        const size_t plen = std::min(std::min(len - off, kFeedPiece), room);
        const char  *piece = sam + off;
        const char  *nl = (const char *)memrchr(piece, '\n', plen);
        uint8_t     *slot = ctx->d_stage[ctx->cur].get();
        if (!nl) {                       // no line ends in this piece: it only grows the carry
            CU(cudaMemcpyAsync(slot + ctx->carry_len, piece, plen, cudaMemcpyHostToDevice, ctx->copy_stream.get()));
            ctx->carry_len += plen;
        } else {
            const size_t cut = (size_t)(nl - piece) + 1, tail = plen - cut;
            CU(cudaMemcpyAsync(slot + ctx->carry_len, piece, cut, cudaMemcpyHostToDevice, ctx->copy_stream.get()));
            int rc = stage_launch(ctx, ctx->carry_len + cut, ctx->fed_bytes + off - ctx->carry_len);
            if (rc != PSSGPU_OK) return rc;
            // (the other buffer is free once the tally that read it, two pieces ago, is done: stage_launch queued the wait)
            if (tail) CU(cudaMemcpyAsync(ctx->d_stage[ctx->cur].get(), piece + cut, tail, cudaMemcpyHostToDevice, ctx->copy_stream.get()));
            ctx->carry_len = tail;
        }
        ctx->h2d_bytes += plen;
        off += plen;
    }
    ctx->fed_bytes += len;
    if (last && ctx->carry_len) {        // final line without '\n' (fgets hands it out as is)
        int rc = stage_launch(ctx, ctx->carry_len, ctx->fed_bytes - ctx->carry_len);
        if (rc != PSSGPU_OK) return rc;
        ctx->carry_len = 0;
    }
    return PSSGPU_OK;
}
}  // namespace

int pssgpu_feed(pssgpu_ctx *ctx, const char *sam, size_t len, int last)
{
    if (!ctx || (!sam && len)) return fail(ctx, PSSGPU_EINVAL, "feed: null argument");
    if (ctx->mode < 0) return fail(ctx, PSSGPU_EINVAL, "feed: no tally open (call *_begin first)");
    Bind bind(ctx);
    const int rc = feed_impl(ctx, sam, len, last);
    // The caller may reuse `sam` as soon as we return -- on success and on every error path alike -- so the copies
    // that read it are waited for.  The tallies are not: they drain at pssgpu_sync / *_finish / get_stats, which is
    // where a kernel fault would surface.  A caller that alternates two pinned buffers (host/pss_host.c) thus
    // overlaps its own reading of the next chunk with the tally of this one.
    const cudaError_t e = cudaStreamSynchronize(ctx->copy_stream.get());
    if (rc != PSSGPU_OK) return rc;
    if (e != cudaSuccess) return fail(ctx, PSSGPU_ECUDA, "feed: %s", cudaGetErrorString(e));
    return PSSGPU_OK;
}

int pssgpu_feed_async(pssgpu_ctx *ctx, const char *sam, size_t len, int last)
{
    if (!ctx || (!sam && len)) return fail(ctx, PSSGPU_EINVAL, "feed_async: null argument");
    if (ctx->mode < 0) return fail(ctx, PSSGPU_EINVAL, "feed_async: no tally open (call *_begin first)");
    Bind bind(ctx);
    const int rc = feed_impl(ctx, sam, len, last);
    if (rc != PSSGPU_OK) cudaStreamSynchronize(ctx->copy_stream.get());      // after an error nothing reads `sam` any more
    return rc;
}

int pssgpu_feed_wait(pssgpu_ctx *ctx)
{
    if (!ctx) return PSSGPU_EINVAL;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->copy_stream.get()));
    return PSSGPU_OK;
}

int pssgpu_feed_device(pssgpu_ctx *ctx, const void *d_sam, size_t len)
{
    if (!ctx || (!d_sam && len)) return fail(ctx, PSSGPU_EINVAL, "feed_device: null argument");
    if (ctx->mode < 0) return fail(ctx, PSSGPU_EINVAL, "feed_device: no tally open (call *_begin first)");
    if (ctx->carry_len) return fail(ctx, PSSGPU_EINVAL, "feed_device: a partial line from pssgpu_feed is pending");
    if ((uintptr_t)d_sam & 15u) return fail(ctx, PSSGPU_EINVAL, "feed_device: pointer must be 16-byte aligned");
    Bind bind(ctx);
    int rc = launch_tally_mode(ctx, (const uint8_t *)d_sam, len, ctx->fed_bytes);
    ctx->fed_bytes += len;
    return rc;
}

int pssgpu_sync(pssgpu_ctx *ctx)
{
    if (!ctx) return PSSGPU_EINVAL;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    { const int brc = bam_check(ctx, false); if (brc != PSSGPU_OK) return brc; }
    time_collect(ctx);
    return PSSGPU_OK;
}

namespace {
// The open tally's pss (which == kModePss) or fragkon table: to the host, its halves to `lo` and `hi`, or, with
// to_device, whole to the device buffer `lo`.
int finish_tally(pssgpu_ctx *ctx, const char *fn, int which, bool to_device, void *lo, void *hi)
{
    if (!ctx || !lo || (!to_device && !hi)) return fail(ctx, PSSGPU_EINVAL, "%s: null argument", fn);
    const bool fk = which == kModeFragkon;
    if (ctx->mode != which && ctx->mode != kModeBoth) return fail(ctx, PSSGPU_EINVAL, "%s: no %s tally open", fn, fk ? "fragkon" : "pss");
    if (ctx->carry_len)
        return fail(ctx, PSSGPU_EINVAL, "%s: %zu bytes of an unterminated line pending (feed with last=1)", fn, ctx->carry_len);
    Bind bind(ctx);
    const size_t half = (fk ? ctx->fk_elems / 2 : (size_t)(ctx->cfg.R + 2) * 16) * sizeof(uint64_t);
    const char  *table = fk ? (const char *)ctx->d_fk.get() : (const char *)ctx->d_tables.get();
    if (to_device) {
        CU(cudaMemcpyAsync(lo, table, 2 * half, cudaMemcpyDeviceToDevice, ctx->stream.get()));
    } else {
        CU(cudaMemcpyAsync(lo, table, half, cudaMemcpyDeviceToHost, ctx->stream.get()));
        CU(cudaMemcpyAsync(hi, table + half, half, cudaMemcpyDeviceToHost, ctx->stream.get()));
    }
    CU(cudaStreamSynchronize(ctx->stream.get()));
    { const int brc = bam_check(ctx, true); if (brc != PSSGPU_OK) return brc; }
    if (!to_device) ctx->d2h_bytes += 2 * half;
    time_collect(ctx);
    return PSSGPU_OK;
}
}  // namespace

int pssgpu_pss_finish(pssgpu_ctx *ctx, uint64_t *fwd, uint64_t *rev) { return finish_tally(ctx, "pss_finish", kModePss, false, fwd, rev); }
int pssgpu_pss_finish_device(pssgpu_ctx *ctx, void *d_tables) { return finish_tally(ctx, "pss_finish_device", kModePss, true, d_tables, nullptr); }
int pssgpu_fragkon_finish(pssgpu_ctx *ctx, uint64_t *fp, uint64_t *tp) { return finish_tally(ctx, "fragkon_finish", kModeFragkon, false, fp, tp); }
int pssgpu_fragkon_finish_device(pssgpu_ctx *ctx, void *d_out)
{
    return finish_tally(ctx, "fragkon_finish_device", kModeFragkon, true, d_out, nullptr);
}

namespace {
int read_stats(pssgpu_ctx *ctx, pssgpu_stats *out, int which)
{
    if (!ctx || !out) return fail(ctx, PSSGPU_EINVAL, "get_stats: null argument");
    if (!ctx->d_stats) return fail(ctx, PSSGPU_EINVAL, "get_stats: no tally was opened");
    Bind bind(ctx);
    unsigned long long h[kStN];
    CU(cudaMemcpyAsync(h, ctx->d_stats.get() + which * kStN, sizeof h, cudaMemcpyDeviceToHost, ctx->stream.get()));
    CU(cudaStreamSynchronize(ctx->stream.get()));
    { const int brc = bam_check(ctx, false); if (brc != PSSGPU_OK) return brc; }
    time_collect(ctx);
    out->lines = h[kStLines];
    out->counted = h[kStCounted];
    out->no_contig = h[kStNoContig];
    out->filtered = h[kStFiltered];
    out->parse_fail = h[kStParseFail];
    out->undefined = h[kStUndefined];
    return PSSGPU_OK;
}
}  // namespace

int pssgpu_get_stats(pssgpu_ctx *ctx, pssgpu_stats *out) { return read_stats(ctx, out, 0); }

int pssgpu_get_fragkon_stats(pssgpu_ctx *ctx, pssgpu_stats *out)
{
    if (ctx && ctx->mode != kModeBoth) return read_stats(ctx, out, 0);      // a fragkon-only tally keeps them in the first set
    return read_stats(ctx, out, 1);
}

// ---- fragkon ------------------------------------------------------------------
void pssgpu_fragkon_default_params(pssgpu_fragkon_params *p)
{
    if (!p) return;
    p->klen = 8;                 // fragkon.c:14
    p->min_mq = 0;               // :15
    p->min_len = 0;              // :16
    p->max_len = 250000000UL;    // :17
    p->merged_only = 0;          // :18
}

// ---- genome-kmer-count ----------------------------------------------------------
int pssgpu_kmer_spectrum_shard_device(pssgpu_ctx *ctx, int k, int shard, int n_shards, void *d_counts)
{
    if (!ctx || !d_counts) return fail(ctx, PSSGPU_EINVAL, "kmer_spectrum: null argument");
    if (!ctx->genome.resident()) return fail(ctx, PSSGPU_ENOGENOME, "kmer_spectrum: no genome resident");
    if (k < 1 || k > kMaxFragK) return fail(ctx, PSSGPU_EUNSUPP, "kmer_spectrum: k %d outside [1,%d]", k, kMaxFragK);
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(ctx, PSSGPU_EINVAL, "kmer_spectrum: shard %d of %d", shard, n_shards);
    Bind bind(ctx);
    const size_t bins = 1ull << (2 * k);
    // k-mers are attributed to the group holding their first base; the last
    // two groups are slack/padding and start no k-mer
    const uint64_t *d_groups = ctx->genome.groups.get();
    const uint64_t usable = ctx->genome.n_groups - 2;
    const uint64_t g0 = usable * (uint64_t)shard / (uint64_t)n_shards;
    const uint64_t g1 = usable * (uint64_t)(shard + 1) / (uint64_t)n_shards;
    const unsigned grid = (unsigned)std::min<uint64_t>(std::max<uint64_t>(1, (g1 - g0 + 255) / 256), (uint64_t)ctx->sm_count * 8);
    // 32-bit bins while no bin can overflow them (fewer than 2^32 positions in the shard)
    // (PSSGPU_SPECTRUM_WIDE: test switch -- run the 64-bit-bin instantiations on a genome that would not need them)
    const bool narrow = (g1 - g0) * 16 < 0xffffffffull && !getenv("PSSGPU_SPECTRUM_WIDE");
    // the scratch buffers of this call are released when it returns, after the stream synchronisation that follows the
    // last launch
    DevPtr<unsigned int> d_narrow;
    if (narrow) {
        CU(alloc(d_narrow, bins * sizeof(unsigned int)));
        cudaError_t e = cudaMemsetAsync(d_narrow.get(), 0, bins * sizeof(unsigned int), ctx->stream.get());
        if (e != cudaSuccess) return fail(ctx, PSSGPU_ECUDA, "kmer_spectrum: %s", cudaGetErrorString(e));
    } else {
        CU(cudaMemsetAsync(d_counts, 0, bins * sizeof(uint64_t), ctx->stream.get()));
    }
    // k = 10 .. 12: radix partition through a scratch buffer (32 bytes per group); without the memory for it, L2 atomics
    DevPtr<uint16_t> d_payload;
    DevPtr<unsigned long long> d_rad;                      // bucket counts | offsets (nb + 1) | cursors
    const uint32_t rad_nb = (k >= 10 && k <= 12) ? (1u << (2 * k - kSpecSmemLog)) : 0u;
    if (rad_nb && g1 > g0) {
        if (alloc(d_payload, (g1 - g0) * 16 * sizeof(uint16_t) + 64) != cudaSuccess
            || alloc(d_rad, (3 * (size_t)rad_nb + 2) * sizeof(unsigned long long)) != cudaSuccess) {
            cudaGetLastError();
            d_payload.reset();
        }
    }
    time_begin(ctx, (g1 - g0) * sizeof(uint64_t));
    // the counting launches, into 32-bit scratch bins or into the caller's 64-bit counters
    auto launch = [&](auto *counts) {
        using CT = std::remove_pointer_t<decltype(counts)>;
        cudaStream_t st = ctx->stream.get();
        if (d_payload) {
            unsigned long long *cnt = d_rad.get(), *off = cnt + rad_nb, *cur = cnt + 2 * (size_t)rad_nb + 1;
            cudaMemsetAsync(cnt, 0, (3 * (size_t)rad_nb + 2) * sizeof(unsigned long long), st);
            const unsigned rgrid = (unsigned)std::min<uint64_t>((g1 - g0 + kRadixThreads - 1) / kRadixThreads, (uint64_t)ctx->sm_count * 4);
            const uint32_t parts = std::max<uint32_t>(1u, (2u * (uint32_t)ctx->sm_count + rad_nb - 1) / rad_nb);
            const size_t   hsmem = (size_t)kSpecSmemBins * sizeof(uint32_t);
            decltype(&radix_count_kernel<10>)   count;
            decltype(&radix_scatter_kernel<10>) scatter;
            switch (k) {
            case 10: count = radix_count_kernel<10>; scatter = radix_scatter_kernel<10>; break;
            case 11: count = radix_count_kernel<11>; scatter = radix_scatter_kernel<11>; break;
            default: count = radix_count_kernel<12>; scatter = radix_scatter_kernel<12>; break;
            }
            count<<<rgrid, kRadixThreads, 0, st>>>(d_groups, g0, g1, cnt);
            radix_scan_kernel<<<1, kRadixThreads, 0, st>>>(cnt, off, cur, rad_nb);
            scatter<<<rgrid, kRadixThreads, 0, st>>>(d_groups, g0, g1, cur, d_payload.get());
            cudaFuncSetAttribute(radix_hist_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem);
            radix_hist_kernel<CT><<<rad_nb * parts, kSpecSmemThreads, hsmem, st>>>(d_payload.get(), off, parts, counts);
        } else if (g1 > g0 && k >= 7 && k <= 9) {
            // shared-memory bins, 16-bit counters packed two to a word: 65 536 bins per CTA -- one pass for 4^8 bins, four for 4^9
            const uint32_t n_slices = (uint32_t)std::min<uint64_t>((uint64_t)ctx->sm_count, (g1 - g0 + kSpecSmemThreads - 1) / kSpecSmemThreads);
            const uint32_t passes = (uint32_t)std::max<size_t>(1, bins >> kSpec16Log);
            const size_t   smem = std::min<size_t>(std::max<size_t>(bins / 2, std::min<size_t>(bins, 32768)), kSpec16Words) * sizeof(uint32_t);
            decltype(&spectrum_smem16_kernel<7, CT>) spec16;
            switch (k) {
            case 7:  spec16 = spectrum_smem16_kernel<7, CT>; break;
            case 8:  spec16 = spectrum_smem16_kernel<8, CT>; break;
            default: spec16 = spectrum_smem16_kernel<9, CT>; break;
            }
            cudaFuncSetAttribute(spec16, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            spec16<<<n_slices * passes, kSpecSmemThreads, smem, st>>>(d_groups, g0, g1, n_slices, counts);
        } else if (g1 > g0) {
            (k <= kSpectrumSmemK ? spectrum_kernel<true, CT> : spectrum_kernel<false, CT>)<<<grid, 256, 0, st>>>(d_groups, g0, g1, k, counts);
        }
    };
    if (narrow) {
        launch(d_narrow.get());
        const unsigned wgrid = (unsigned)std::min<uint64_t>((bins + 255) / 256, (uint64_t)ctx->sm_count * 8);
        widen_kernel<<<wgrid, 256, 0, ctx->stream.get()>>>(d_narrow.get(), (unsigned long long *)d_counts, bins);
    } else {
        launch((unsigned long long *)d_counts);
    }
    time_end(ctx);
    cudaError_t le = cudaGetLastError();
    cudaError_t se = cudaStreamSynchronize(ctx->stream.get());
    if (le != cudaSuccess || se != cudaSuccess)
        return fail(ctx, PSSGPU_ECUDA, "kmer_spectrum: %s", cudaGetErrorString(le != cudaSuccess ? le : se));
    time_collect(ctx);
    return PSSGPU_OK;
}

int pssgpu_kmer_spectrum_shard(pssgpu_ctx *ctx, int k, int shard, int n_shards, uint64_t *counts)
{
    if (!ctx || !counts) return fail(ctx, PSSGPU_EINVAL, "kmer_spectrum: null argument");
    if (k < 1 || k > kMaxFragK) return fail(ctx, PSSGPU_EUNSUPP, "kmer_spectrum: k %d outside [1,%d]", k, kMaxFragK);
    Bind bind(ctx);
    const size_t bins = 1ull << (2 * k);
    DevPtr<uint64_t> d;
    CU(alloc(d, bins * sizeof(uint64_t)));
    int rc = pssgpu_kmer_spectrum_shard_device(ctx, k, shard, n_shards, d.get());
    if (rc == PSSGPU_OK) {
        cudaError_t e = cudaMemcpy(counts, d.get(), bins * sizeof(uint64_t), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(ctx, PSSGPU_ECUDA, "kmer_spectrum: D2H: %s", cudaGetErrorString(e));
        else ctx->d2h_bytes += bins * sizeof(uint64_t);
    }
    return rc;
}

int pssgpu_kmer_spectrum(pssgpu_ctx *ctx, int k, uint64_t *counts) { return pssgpu_kmer_spectrum_shard(ctx, k, 0, 1, counts); }

// ---- measurement hooks ------------------------------------------------------------
int pssgpu_timing_reset(pssgpu_ctx *ctx, int enable)
{
    if (!ctx) return PSSGPU_EINVAL;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    time_collect(ctx);
    ctx->timing = enable != 0;
    ctx->launches = ctx->bytes_scanned = ctx->h2d_bytes = ctx->d2h_bytes = 0;
    ctx->kernel_ms = 0.0;
    return PSSGPU_OK;
}

int pssgpu_timing_get(pssgpu_ctx *ctx, pssgpu_timing *out)
{
    if (!ctx || !out) return PSSGPU_EINVAL;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    time_collect(ctx);
    out->launches = ctx->launches;
    out->kernel_ms = ctx->kernel_ms;
    out->bytes_scanned = ctx->bytes_scanned;
    out->h2d_bytes = ctx->h2d_bytes;
    out->d2h_bytes = ctx->d2h_bytes;
    return PSSGPU_OK;
}

// ---- test hook -------------------------------------------------------------------------
int pssgpu_debug_status(pssgpu_ctx *ctx, int enable)
{
    if (!ctx) return PSSGPU_EINVAL;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    if (enable && !ctx->dbg_cap) {               // (after a call that failed half way, everything is allocated again)
        const uint64_t cap = 8ull << 20;
        CU(alloc(ctx->d_dbg_off, cap * sizeof(uint64_t)));
        CU(alloc(ctx->d_dbg_code, cap));
        CU(alloc(ctx->d_dbg_n, sizeof(unsigned long long)));
        CU(cudaMemset(ctx->d_dbg_n.get(), 0, sizeof(unsigned long long)));
        ctx->dbg_cap = cap;
    }
    ctx->dbg = enable != 0;
    return PSSGPU_OK;
}

int pssgpu_debug_fetch(pssgpu_ctx *ctx, uint64_t *offsets, int8_t *codes, uint64_t cap, uint64_t *n)
{
    if (!ctx || !n) return PSSGPU_EINVAL;
    *n = 0;
    if (!ctx->dbg_cap) return PSSGPU_OK;
    Bind bind(ctx);
    CU(cudaStreamSynchronize(ctx->stream.get()));
    unsigned long long have = 0;
    CU(cudaMemcpy(&have, ctx->d_dbg_n.get(), sizeof have, cudaMemcpyDeviceToHost));
    if (have > ctx->dbg_cap) have = ctx->dbg_cap;
    const uint64_t take = std::min<uint64_t>(have, cap);
    if (take && offsets) CU(cudaMemcpy(offsets, ctx->d_dbg_off.get(), take * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (take && codes) CU(cudaMemcpy(codes, ctx->d_dbg_code.get(), take, cudaMemcpyDeviceToHost));
    *n = take;
    return PSSGPU_OK;
}

}  // extern "C"
