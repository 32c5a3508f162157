// C ABI of tagdigger_b200 (see include/tagdigger_b200.h): contexts, table
// upload, chunk streaming with pinned buffers, zlib inflate on a host thread.
// There is no CPU counting path in this file: every count comes from
// count_kernel (tdg_kernel.cuh), or from split_count / split_count_batch
// (tdg_split.cuh) when the splitter's trimmed reads are counted.
#include <cuda_runtime.h>
#include <zlib.h>

#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/tagdigger_b200.h"
#include "tdg_kernel.cuh"
#include "tdg_csv.h"
#include "tdg_comm.h"
#include "tdg_feed.h"
#include "tdg_text.h"
#include "tdg_tables.h"
#include "tdg_trim.cuh"
#include "tdg_split.cuh"
#include "tdg_gzchain.h"
#include "tdg_gzdev.cuh"
#include "tdg_bgzf.cuh"

static_assert(TDG_HALO_BYTES >= tdg::HALO, "the allocation slack promised by the header must cover the kernel halo");
static_assert(TDG_TILE_BYTES >= tdg::TILE, "the allocation granule promised by the header must cover a kernel tile");

namespace {

constexpr int NSLOT = 3;
constexpr int MAX_TIMED = 4096;
std::string g_create_error;

// A device or pinned buffer of the context.  Allocated by reserve() (below), freed by its destructor.
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    bool host = false;

    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    Buf(Buf &&o) noexcept : p(o.p), cap(o.cap), host(o.host) { o.p = nullptr, o.cap = 0; }
    Buf &operator=(Buf &&o) noexcept
    {
        if (this != &o) {
            reset();
            p = o.p, cap = o.cap, host = o.host;
            o.p = nullptr, o.cap = 0;
        }
        return *this;
    }
    ~Buf() { reset(); }
    void reset()
    {
        if (p) {
            if (host) cudaFreeHost(p); else cudaFree(p);
        }
        p = nullptr;
        cap = 0;
    }
};

// An event of the context.  Created on first use by make_event() (below), destroyed by its destructor.
struct Event {
    cudaEvent_t e = nullptr;

    Event() = default;
    Event(const Event &) = delete;
    Event &operator=(const Event &) = delete;
    Event(Event &&o) noexcept : e(o.e) { o.e = nullptr; }
    ~Event()
    {
        if (e) cudaEventDestroy(e);
    }
    operator cudaEvent_t() const { return e; }
};

struct Slot {
    Buf dev;
    Buf carry;       // pinned: partial last line of the previous piece
    Event copied;    // H2D of this slot finished
    Event done;      // kernel on this slot finished
};

}  // namespace

// how the host feeder continues when the device gzip feed stops early (tdg_gzdev.cuh)
struct GzHandover {
    bool active = false;
    bool to_zlib = false;
    bool bgzf = false;           // BGZF: the host feeder continues at the member at file offset bgzf_off
    uint64_t bgzf_off = 0;
    uint64_t pos_bit = 0, member_len = 0, delivered = 0;
    uint32_t hist = 0, crc = 0;
    std::vector<uint8_t> window;
};

// The host feeder of `path`: from the start, or where the device gzip feed handed over (ho->active)
static int open_feed(tdg::Feeder &feed, const char *path, bool gz, const GzHandover *ho)
{
    if (!ho || !ho->active) return feed.open(path, gz);
    if (ho->bgzf) return feed.open_resume_bgzf(path, ho->bgzf_off, ho->delivered);
    return feed.open_resume(path, ho->pos_bit, ho->to_zlib ? nullptr : ho->window.data(), ho->hist, ho->crc, ho->member_len,
                            ho->delivered);
}

// The host side of tdg_count_file for one file: a thread that reads (or inflates) the file through
// tdg_feed.h into three pinned buffers, one ahead of the other.  It can be started BEFORE its
// file's turn (the `next_path` of tdg_count_file2): a key of many small files then never waits for
// a read -- the next file's bytes arrive while this file's are copied and counted.
struct FileReader {
    static constexpr int NBUF = 3;
    struct Buf {
        uint8_t *p = nullptr;
        size_t n = 0;
        int state = 0;          // 0 free, 1 full
        bool high = false;      // some byte >= 0x80: the text needs UTF-8 validation
        int err = 0;            // the read that should have filled this buffer failed
        std::string msg;
    } bufs[NBUF];
    std::mutex mu;
    std::condition_variable cv;
    bool stop = false;
    std::thread th;
    std::string path;
    bool gz = false;
    size_t chunk = 0;
    int set = 0;                // which of the context's two sets of pinned buffers it fills
    GzHandover ho;

    void start()
    {
        th = std::thread([this]() {
            // host feed: parallel pread / parallel BGZF inflate / zlib, see tdg_feed.h
            tdg::Feeder feed;
            int orc = open_feed(feed, path.c_str(), gz, &ho);
            int bi = 0;
            for (;;) {
                Buf &b = bufs[bi];
                {
                    std::unique_lock<std::mutex> lk(mu);
                    cv.wait(lk, [&] { return b.state == 0 || stop; });
                    if (stop) break;
                }
                long long r = orc ? orc : feed.fill(b.p, chunk);
                size_t got = 0;
                int err = 0;
                std::string msg;
                if (r < 0) { err = (int)r; msg = feed.error(); }
                else got = (size_t)r;
                const bool high = got ? tdg::has_high_bit_mt(b.p, got, feed.threads()) : false;
                {
                    std::lock_guard<std::mutex> lk(mu);
                    b.n = got;
                    b.high = high;
                    b.err = err;
                    b.msg = msg;
                    b.state = 1;
                }
                cv.notify_all();
                if (got == 0 || err) break;           // end of file, or the defect: nothing comes after it
                bi = (bi + 1) % NBUF;
            }
        });
    }
    ~FileReader()
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv.notify_all();
        if (th.joinable()) th.join();
    }
};

struct tdg_ctx {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;          // dynamic shared memory a block of the counting kernel may use
    std::string err;
    size_t chunk_bytes = 0;

    cudaStream_t stream = nullptr;       // kernels
    cudaStream_t copy_stream = nullptr;  // H2D
    Event handoff;                       // tdg_stream_wait / tdg_other_stream_wait

    // tables
    tdg::HostTagTable tags;
    bool have_tags = false;
    Buf d_entries, d_ext;                // TagEntry[], uint64_t[]
    std::vector<uint8_t> bar_blob;
    bool have_bar = false;
    Buf d_bar;

    // matrix: the context's own (tdg_set_matrix) or the caller's (tdg_bind_matrix)
    int32_t *d_matrix = nullptr;
    Buf matrix;
    uint32_t rows = 0, cols = 0;
    uint32_t max_row = 0, max_col = 0;   // largest indices the loaded tables refer to
    // extra zero-initialised copies of a small matrix (see ChunkArgs::replicas); always all-zero between launches
    Buf d_replicas;
    uint32_t n_replicas = 1;

    // per-launch scratch (ScratchHeader, SegInfo[], FixEntry[])
    Buf d_sync;
    int occ[3] = {0, 0, 0};              // resident CTAs per SM of the three kernel instantiations, at
    size_t occ_smem[3] = {0, 0, 0};      //   this much dynamic shared memory
    uint32_t force_seg_tiles = 0; // test hook (TDG_SEG_TILES)
    bool force_general = false;   // test hook (TDG_GENERAL=1): never use the fast matcher
    Buf d_state;                  // LineState[2]
    int state_cur = 0;
    Buf d_totals;                 // unsigned long long[4]

    // streaming
    Slot slot[NSLOT];
    bool have_slots = false;
    int next_slot = 0;
    size_t carry_len = 0;        // bytes waiting in slot[next_slot].carry
    bool file_open = false;

    // trim decision tables (tdg_set_trim): one device blob
    Buf d_trim;
    tdg::TrimArgs trim;          // device pointers into d_trim
    uint32_t trim_nbar = 0;
    bool have_trim = false;

    // staging of tdg_trim_batch, tdg_split_batch and tdg_match_batch
    Buf batch;

    // streaming splitter (tdg_split_begin / tdg_split_block): growable device and pinned buffers
    Buf sp_in, sp_tiles, sp_ends, sp_rec, sp_flags, sp_sums, sp_base, sp_out, sp_tabs;      // device
    Buf sp_hout, sp_hflags, sp_hbase;                                                          // pinned host
    uint32_t sp_nbar = 0, sp_cutlen = 0;
    bool have_split = false;

    // counting the splitter's records instead of writing them (tdg_split_count_*): the stage-2 barcode
    // table, the matrix row of every stage-1 barcode, and a block's totals [4] + complex flag
    Buf sc_bar, sc_rows, sc_tot;         // device
    Buf sc_htot;                         // pinned host
    uint32_t sc_max_row = 0;
    bool have_split_count = false;

    // BGZF output of the splitter (tdg_split_bgzf, tdg_bgzf.cuh): every barcode's pending tail
    // (< 65,280 bytes) waits in bz_tail between calls
    bool bz_on = false, bz_attr = false;
    Buf bz_tail, bz_src, bz_mem, bz_copy, bz_match, bz_work, bz_size, bz_out;      // device
    Buf bz_hmem, bz_hcopy, bz_hsize, bz_hout;                                     // pinned host
    std::vector<uint32_t> bz_tail_len;
    std::vector<uint64_t> bz_off;
    uint32_t bz_op[8] = {0, 0, 0, 0, 0, 0, 0, 0};

    // pinned buffers of tdg_count_file (kept between files: pinning 192 MiB costs ~0.1 s), chunk_bytes each;
    // set 1 is for the reader that runs ahead for the next file
    Buf file_buf[2][FileReader::NBUF];
    std::unique_ptr<FileReader> ahead;                        // started by tdg_count_file2's next_path

    // device-side gzip feed (tdg_gzdev.cuh): growable buffers, kept between files
    Buf gz_comp, gz_comp2, gz_syms, gz_sym2, gz_ntok, gz_meta, gz_cand, gz_ncand, gz_windows, gz_text, gz_crc, gz_lens, gz_offs, gz_tabs, gz_carry, gz_cold;   // device
    Buf gz_hmeta, gz_hcrc, gz_htail;                                                                                       // pinned host
    Event gz_up[3];
    Event gz_pre;
    int64_t last_file[3] = {0, 0, 0};    // tdg_count_file: device gzip rounds, chunks accepted, 0 all on the device / 1 host feeder took over / -1 host feeder only
    bool gz_tables = false;
    uint32_t gz_op[8] = {0, 0, 0, 0, 0, 0, 0, 0};

    // multi-GPU: the communicator of tdg_comm_init (one rank per context)
    tdg::NcclApi::Comm comm = nullptr;
    int comm_ranks = 1;

    // accounting
    uint64_t launches = 0;
    bool timing = false;
    std::vector<Event> tev;      // 2 * MAX_TIMED
    int tev_used = 0;

    // test hook (TDG_FAIL_ALLOC=k): the k-th buffer allocation or event creation after tdg_create fails
    uint64_t fail_at = 0, allocs = 0;
};

namespace {

int fail(tdg_ctx *ctx, int code, const std::string &msg)
{
    if (ctx) ctx->err = msg; else g_create_error = msg;
    return code;
}

#define CK(call)                                                                                 \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail(ctx, TDG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

bool simulated_failure(tdg_ctx *ctx) { return ctx->fail_at && ++ctx->allocs == ctx->fail_at; }

// Every buffer of the context comes from here: when b holds fewer than `need` bytes, it is replaced by
// a buffer of `cap` bytes (contents are NOT kept).  The old buffer is freed only once the new one is
// had, so it stays whole when the allocation fails.
int reserve(tdg_ctx *ctx, Buf &b, size_t need, size_t cap, bool host)
{
    if (need <= b.cap) return TDG_OK;
    CK(cudaStreamSynchronize(ctx->stream));
    void *fresh = nullptr;
    const bool sim = simulated_failure(ctx);
    cudaError_t e = sim ? cudaErrorMemoryAllocation : host ? cudaHostAlloc(&fresh, cap, cudaHostAllocDefault) : cudaMalloc(&fresh, cap);
    if (e != cudaSuccess) {
        cudaGetLastError();                                  // (the failed allocation must not show up as the next launch's error)
        return fail(ctx, TDG_ERR_NOMEM, std::string("buffer of ") + std::to_string(cap) + " bytes: " +
                                            (sim ? "simulated (TDG_FAIL_ALLOC)" : cudaGetErrorString(e)));
    }
    b.reset();
    b.p = fresh;
    b.cap = cap;
    b.host = host;
    return TDG_OK;
}

// growable buffers: a quarter more than asked for
int grow(tdg_ctx *ctx, Buf &b, size_t need, bool host) { return reserve(ctx, b, need, need + need / 4 + 4096, host); }
int grow_exact(tdg_ctx *ctx, Buf &b, size_t need, bool host) { return reserve(ctx, b, need, need, host); }

int make_event(tdg_ctx *ctx, Event &ev, unsigned flags = cudaEventDisableTiming)
{
    if (ev.e) return TDG_OK;
    if (simulated_failure(ctx)) return fail(ctx, TDG_ERR_NOMEM, "event: simulated (TDG_FAIL_ALLOC)");
    CK(cudaEventCreateWithFlags(&ev.e, flags));
    return TDG_OK;
}

// per-launch scratch: header, then SegInfo[num_segs], then FixEntry[num_segs]
struct ScratchHeader {
    unsigned long long ticket_main, ticket_fix;
    uint32_t n_fix, last_kind;
    unsigned long long pad;
    unsigned long long run_total[32 * 32];      // verify_sums -> verify_kernel (VERIFY_MAX_CTAS runs of 32 warps)
};
static_assert(offsetof(ScratchHeader, run_total) == 32, "scratch header layout");
static_assert(sizeof(ScratchHeader::run_total) / 8 == tdg::VERIFY_MAX_CTAS * (tdg::VERIFY_THREADS / 32), "one total per run");

int ensure_sync(tdg_ctx *ctx, size_t segs)
{
    size_t need = (sizeof(ScratchHeader) + segs * (sizeof(tdg::SegInfo) + sizeof(tdg::FixEntry)) + 7) / 8;     // 8-byte words
    return reserve(ctx, ctx->d_sync, need * 8, (need + need / 2) * 8, false);
}

// tdg_timing_begin: a pair of events around the launches of one call, on ctx->stream.  Both are created
// (on first use) before the first is recorded; the caller records the second behind its launches.
int timed_start(tdg_ctx *ctx, bool &timed)
{
    timed = ctx->timing && ctx->tev_used + 2 <= MAX_TIMED * 2;
    if (!timed) return TDG_OK;
    int rc;
    if ((rc = make_event(ctx, ctx->tev[ctx->tev_used], cudaEventDefault)) || (rc = make_event(ctx, ctx->tev[ctx->tev_used + 1], cudaEventDefault)))
        return rc;
    CK(cudaEventRecord(ctx->tev[ctx->tev_used++], ctx->stream));
    return TDG_OK;
}

typedef void (*CountKernel)(const tdg::ChunkArgs);

// The three instantiations of the counting kernel: scan only, the matcher for tags that fit the
// 128-bit key, and its long form (tags of up to 160 bases: key + 96 bases of tail).
CountKernel pick_kernel(bool match, bool long_tags)
{
    if (!match) return tdg::count_kernel<false, false>;
    return long_tags ? tdg::count_kernel<true, true> : tdg::count_kernel<true, false>;
}

int kernel_geometry(tdg_ctx *ctx, CountKernel kern, size_t smem, int *per_sm)
{
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kern, tdg::THREADS, smem));
    if (*per_sm < 1) return fail(ctx, TDG_ERR_CUDA, "counting kernel does not fit on an SM");
    return TDG_OK;
}

template <bool MATCH>
int launch_chunk(tdg_ctx *ctx, const void *dev_bytes, size_t n, uint64_t line_base, int prev_kind,
                 uint64_t reads_limit)
{
    using namespace tdg;
    if (n == 0) return TDG_OK;
    if (((uintptr_t)dev_bytes & 15u) != 0) return fail(ctx, TDG_ERR_ARG, "device chunk must be 16-byte aligned");
    size_t tiles = (n + TILE - 1) / TILE;
    if (tiles >= 0xFFFFFFFFull) return fail(ctx, TDG_ERR_ARG, "chunk too large (limit 2^32 - 2 tiles)");

    size_t bar_smem = 0;
    if (MATCH && ctx->bar_blob.size() <= BAR_SMEM_MAX) bar_smem = round_up(ctx->bar_blob.size(), 16);
    if (SMEM_FIXED + bar_smem > ctx->smem_optin) bar_smem = 0;      // no room: the kernel reads the table from global memory
    size_t smem = SMEM_FIXED + bar_smem;
    uint32_t fast_words = 0;
    bool long_tags = false;
    if (MATCH) {
        fast_words = ctx->force_general ? 0 : fast_words_for((const BarTable *)ctx->bar_blob.data(), ctx->tags.t);
        long_tags = fast_words != 0 && fast_is_long(ctx->tags.t);
    }
    const CountKernel kern = pick_kernel(MATCH, long_tags);
    const int ki = !MATCH ? 0 : (long_tags ? 2 : 1);
    int &per_sm = ctx->occ[ki];
    size_t &occ_smem = ctx->occ_smem[ki];
    if (per_sm == 0 || occ_smem != smem) {
        int rc = kernel_geometry(ctx, kern, smem, &per_sm);
        if (rc) return rc;
        occ_smem = smem;
    }
    size_t max_grid = (size_t)per_sm * ctx->sm_count;
    size_t workers = max_grid * WARPS;      // every warp is an independent pipeline
    // Segments: runs of consecutive tiles handed to one warp through the ticket counter.  Long
    // ones (about 16 per warp, at most 64 tiles: a segment start costs a ticket, a structure guess
    // and -- when the guess is wrong -- a redo of the whole segment) for the first 7/8 of the
    // launch, eight times shorter ones for the rest, so that the warps finish together.
    size_t seg_tiles = tiles / (workers * 16);
    if (seg_tiles < 1) seg_tiles = 1;
    if (seg_tiles > 64) seg_tiles = 64;
    size_t seg_small = seg_tiles / 8 ? seg_tiles / 8 : 1;
    if (ctx->force_seg_tiles) seg_tiles = seg_small = ctx->force_seg_tiles;
    size_t n_big = tiles / seg_tiles * 7 / 8;
    size_t rest = tiles - n_big * seg_tiles;
    size_t segs = n_big + (rest + seg_small - 1) / seg_small;
    size_t grid = (segs + WARPS - 1) / WARPS;
    if (grid > max_grid) grid = max_grid;

    int rc = ensure_sync(ctx, segs);
    if (rc) return rc;
    ScratchHeader *hdr = (ScratchHeader *)ctx->d_sync.p;
    SegInfo *seginfo = (SegInfo *)(hdr + 1);
    FixEntry *fix = (FixEntry *)(seginfo + segs);
    CK(cudaMemsetAsync(hdr, 0, offsetof(ScratchHeader, run_total), ctx->stream));

    ChunkArgs a;
    memset(&a, 0, sizeof(a));
    a.bytes = (const uint8_t *)dev_bytes;
    a.n = n;
    a.num_tiles = (uint32_t)tiles;
    a.seg_tiles = (uint32_t)seg_tiles;
    a.n_big = (uint32_t)n_big;
    a.seg_small = (uint32_t)seg_small;
    a.num_segs = (uint32_t)segs;
    a.mode = MODE_MAIN;
    VerifyArgs v;
    memset(&v, 0, sizeof(v));
    if (line_base == TDG_LINE_CHAINED) {
        a.use_arg_state = v.use_arg_state = 0;
    } else {
        a.use_arg_state = v.use_arg_state = 1;
        a.line_base = v.line_base = line_base;
        a.prev_kind = v.prev_kind = (uint32_t)prev_kind;
    }
    LineState *state = (LineState *)ctx->d_state.p;
    a.state_in = v.state_in = state + ctx->state_cur;
    v.state_out = state + (ctx->state_cur ^ 1);
    ctx->state_cur ^= 1;
    a.ticket = &hdr->ticket_main;
    a.seginfo = seginfo;
    a.last_kind = &hdr->last_kind;
    a.fix = fix;
    a.n_fix = &hdr->n_fix;
    a.reads_limit = reads_limit;
    a.halo_bytes = HALO;
    if (MATCH) {
        const BarTable *hbar = (const BarTable *)ctx->bar_blob.data();
        a.fast_words = fast_words;
        if (a.fast_words) {
            // the fast matcher reads whole 4-word groups from the aligned word of the line start
            uint32_t need = hbar->max_tag_off + ctx->tags.t.max_len + 36u;
            uint32_t touch = 4u * a.fast_words + 16u;
            uint32_t h = (std::max(need, touch) + 15u) & ~15u;
            a.halo_bytes = std::min<uint32_t>(std::max<uint32_t>(h, 128u), HALO);
        }
        {
            // uniform matcher constants, computed once here instead of by every thread
            const TagTable &tt = ctx->tags.t;
            a.need = std::max<uint32_t>(hbar->max_tag_off + tt.max_len, hbar->max_len) + 36u;
            a.tag_km = lowmask(tt.cls[0].K);
            if (tt.min_len == tt.max_len && tt.max_len <= 64) {
                a.ulen = tt.max_len;
                for (uint32_t k = 0; k < 4; k++) {
                    uint32_t nb = a.ulen > 16 * k ? a.ulen - 16 * k : 0;
                    a.um[k] = nb >= 16 ? 0xFFFFFFFFu : ((1u << (2 * nb)) - 1u);
                }
            }
        }
        a.bar = (const BarTable *)ctx->d_bar.p;
        a.bar_bytes = (uint32_t)ctx->bar_blob.size();
        a.bar_in_smem = bar_smem != 0;
        a.cols = ctx->cols;
        a.tags = ctx->tags.t;
        a.tags.entries = (const TagEntry *)ctx->d_entries.p;
        a.tags.ext = (const uint64_t *)ctx->d_ext.p;
        a.matrix = ctx->d_matrix;
        a.replicas = (int32_t *)ctx->d_replicas.p;
        a.n_replicas = ctx->n_replicas;
        a.cells = ctx->rows * ctx->cols;
        a.totals = (unsigned long long *)ctx->d_totals.p;
    }
    v.num_segs = (uint32_t)segs;
    v.make_fixes = MATCH ? 1 : 0;
    v.reads_limit = reads_limit;
    v.seginfo = seginfo;
    v.last_kind = &hdr->last_kind;
    v.fix = fix;
    v.n_fix = &hdr->n_fix;
    v.run_total = hdr->run_total;

    bool timed;
    if ((rc = timed_start(ctx, timed))) return rc;
    kern<<<(unsigned)grid, THREADS, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    // every warp of the verify launches takes >= 256 segments
    const unsigned vgrid = (unsigned)std::min<size_t>(VERIFY_MAX_CTAS, std::max<size_t>(1, segs / (32 * 256)));
    verify_sums<<<vgrid, VERIFY_THREADS, 0, ctx->stream>>>(v);
    CK(cudaGetLastError());
    verify_kernel<<<vgrid, VERIFY_THREADS, 0, ctx->stream>>>(v);
    CK(cudaGetLastError());
    ctx->launches += 3;
    if (MATCH) {
        // redo mis-numbered segments (none for well-formed FASTQ: the CTAs exit at once)
        a.mode = MODE_FIX;
        a.ticket = &hdr->ticket_fix;
        size_t fgrid = 2 * segs < max_grid ? 2 * segs : max_grid;
        kern<<<(unsigned)fgrid, THREADS, smem, ctx->stream>>>(a);
        CK(cudaGetLastError());
        ctx->launches += 1;
        if (ctx->n_replicas > 1) {
            unsigned fold_grid = (unsigned)std::min<size_t>(((size_t)a.cells + 255) / 256, (size_t)ctx->sm_count * 8);
            fold_kernel<<<fold_grid, 256, 0, ctx->stream>>>(ctx->d_matrix, a.replicas, a.cells, ctx->n_replicas - 1);
            CK(cudaGetLastError());
            ctx->launches += 1;
        }
    }
    if (timed) CK(cudaEventRecord(ctx->tev[ctx->tev_used++], ctx->stream));
    return TDG_OK;
}

// Small matrices get up to 16 copies (<= 4 MiB in total) that the warps update in turn;
// fold_kernel adds them up after every launch.  With few rows (pre-split files: ONE row)
// the most frequent tags would otherwise serialise all SMs on a handful of L2 addresses.
int size_replicas(tdg_ctx *ctx)
{
    size_t cells = (size_t)ctx->rows * ctx->cols;
    size_t bytes = cells * sizeof(int32_t);
    uint32_t want = 1;
    if (bytes && bytes <= ((size_t)2 << 20)) want = (uint32_t)std::min<size_t>(16, ((size_t)4 << 20) / bytes);
    if (const char *e = getenv("TDG_REPLICAS")) want = (uint32_t)std::max(1, atoi(e));
    ctx->n_replicas = 1;
    if (want > 1) {
        size_t need = (size_t)(want - 1) * cells * sizeof(int32_t);
        int rc = grow_exact(ctx, ctx->d_replicas, need, false);
        if (rc) return rc;
        CK(cudaMemsetAsync(ctx->d_replicas.p, 0, need, ctx->stream));
        ctx->n_replicas = want;
    }
    return TDG_OK;
}

int need_device(tdg_ctx *ctx)
{
    if (!ctx) return TDG_ERR_ARG;
    return TDG_OK;
}

int need_ready(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_tags) return fail(ctx, TDG_ERR_STATE, "tdg_set_tags has not been called");
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "tdg_set_matrix / tdg_bind_matrix has not been called");
    if (!ctx->have_bar) return fail(ctx, TDG_ERR_STATE, "tdg_begin_file has not been called");
    if (ctx->max_col >= ctx->cols) return fail(ctx, TDG_ERR_ARG, "a tag column lies outside the matrix");
    if (ctx->max_row >= ctx->rows) return fail(ctx, TDG_ERR_ARG, "a barcode row lies outside the matrix");
    return TDG_OK;
}

int ensure_slots(tdg_ctx *ctx)
{
    if (ctx->have_slots) return TDG_OK;
    // a piece is the carried partial line (<= chunk_bytes) plus up to chunk_bytes new bytes
    size_t cap = round_up(2 * ctx->chunk_bytes, TDG_TILE_BYTES) + TDG_TILE_BYTES + TDG_HALO_BYTES;
    for (Slot &s : ctx->slot) {
        int rc;
        if ((rc = grow_exact(ctx, s.dev, cap, false)) || (rc = grow_exact(ctx, s.carry, 1 << 20, true)) ||
            (rc = make_event(ctx, s.copied)) || (rc = make_event(ctx, s.done)))
            return rc;
    }
    ctx->have_slots = true;
    return TDG_OK;
}

// a slot's carry doubles until it holds `need` bytes, and keeps its first `keep`
int grow_carry(tdg_ctx *ctx, Buf &carry, size_t need, size_t keep)
{
    if (need <= carry.cap) return TDG_OK;
    size_t cap = carry.cap;
    while (cap < need) cap *= 2;
    Buf fresh;
    int rc = grow_exact(ctx, fresh, cap, true);
    if (rc) return rc;
    if (keep) memcpy(fresh.p, carry.p, keep);
    carry = std::move(fresh);
    return TDG_OK;
}

// Where to cut bytes[0..n) so that everything before the cut is whole lines:
// just after the last '\n', or (files with lone '\r' line ends) after the last
// '\r' that is followed by another byte which is not '\n'.  0 if no line ends.
size_t line_cut(const uint8_t *b, size_t n)
{
    const void *lf = memrchr(b, '\n', n);
    size_t cut = lf ? (size_t)((const uint8_t *)lf - b) + 1 : 0;
    // a lone '\r' after that point ends a line too
    if (cut < n) {
        const uint8_t *tail = b + cut;
        size_t m = n - cut;
        for (size_t i = m; i-- > 0;) {
            if (tail[i] == '\r' && i + 1 < m) {      // tail[i+1] cannot be '\n' (it lies after the last '\n')
                cut += i + 1;
                break;
            }
        }
    }
    return cut;
}

// One piece: [carry | bytes[0..cut)] -> device slot -> kernel; bytes[cut..n) becomes the new carry.
int submit_piece(tdg_ctx *ctx, const uint8_t *bytes, size_t n, size_t cut, uint64_t reads_limit)
{
    int si = ctx->next_slot;
    Slot &s = ctx->slot[si];
    size_t total = ctx->carry_len + cut;
    int nxt = (si + 1) % NSLOT;
    Slot &sn = ctx->slot[nxt];
    if (cut > 0) {      // the piece holds a line end: carried bytes + everything up to the cut form whole lines
        // the slot's previous kernel must be finished before its buffer is overwritten
        CK(cudaStreamWaitEvent(ctx->copy_stream, s.done, 0));
        uint8_t *dev = (uint8_t *)s.dev.p;
        if (ctx->carry_len) CK(cudaMemcpyAsync(dev, s.carry.p, ctx->carry_len, cudaMemcpyHostToDevice, ctx->copy_stream));
        if (cut) CK(cudaMemcpyAsync(dev + ctx->carry_len, bytes, cut, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(s.copied, ctx->copy_stream));
        CK(cudaStreamWaitEvent(ctx->stream, s.copied, 0));
        int rc = launch_chunk<true>(ctx, dev, total, TDG_LINE_CHAINED, 0, reads_limit);
        if (rc) return rc;
        CK(cudaEventRecord(s.done, ctx->stream));
        // new carry goes to the next slot's pinned buffer, once its last H2D has drained
        CK(cudaEventSynchronize(sn.copied));
        size_t rest = n - cut;
        int rc2 = grow_carry(ctx, sn.carry, rest, 0);
        if (rc2) return rc2;
        if (rest) memcpy(sn.carry.p, bytes + cut, rest);
        ctx->carry_len = rest;
        ctx->next_slot = nxt;
    } else {
        // nothing complete yet: append to the current carry
        size_t rest = n;
        if (ctx->carry_len + rest > ctx->chunk_bytes)
            return fail(ctx, TDG_ERR_ARG, "a single text line is longer than chunk_bytes");
        int rc2 = grow_carry(ctx, s.carry, ctx->carry_len + rest, ctx->carry_len);
        if (rc2) return rc2;
        memcpy((uint8_t *)s.carry.p + ctx->carry_len, bytes, rest);
        ctx->carry_len += rest;
    }
    return TDG_OK;
}

int submit_impl(tdg_ctx *ctx, const uint8_t *bytes, size_t n, uint64_t reads_limit, bool wait_copied)
{
    int rc = ensure_slots(ctx);
    if (rc) return rc;
    size_t pos = 0;
    int last = -1;
    static const bool sdebug = getenv("TDG_FILE_DEBUG") != nullptr;
    const auto s0 = std::chrono::steady_clock::now();
    while (pos < n) {
        size_t m = n - pos < ctx->chunk_bytes ? n - pos : ctx->chunk_bytes;
        size_t cut = line_cut(bytes + pos, m);
        if (ctx->carry_len + cut > 2 * ctx->chunk_bytes)
            return fail(ctx, TDG_ERR_ARG, "a single text line is longer than chunk_bytes");
        if (cut) last = ctx->next_slot;
        rc = submit_piece(ctx, bytes + pos, m, cut, reads_limit);
        if (rc) return rc;
        pos += m;
    }
    const auto s1 = std::chrono::steady_clock::now();
    if (wait_copied && last >= 0) CK(cudaEventSynchronize(ctx->slot[last].copied));
    if (sdebug)
        fprintf(stderr, "  submit %zu bytes: enqueue %.2f ms, wait for the copy %.2f ms\n", n,
                std::chrono::duration<double, std::milli>(s1 - s0).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - s1).count());
    return TDG_OK;
}

int end_file_impl(tdg_ctx *ctx, uint64_t reads_limit)
{
    if (ctx->carry_len) {
        // the carried bytes are the file's last line (no line end follows)
        int si = ctx->next_slot;
        Slot &s = ctx->slot[si];
        CK(cudaStreamWaitEvent(ctx->copy_stream, s.done, 0));
        CK(cudaMemcpyAsync(s.dev.p, s.carry.p, ctx->carry_len, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(s.copied, ctx->copy_stream));
        CK(cudaStreamWaitEvent(ctx->stream, s.copied, 0));
        int rc = launch_chunk<true>(ctx, s.dev.p, ctx->carry_len, TDG_LINE_CHAINED, 0, reads_limit);
        if (rc) return rc;
        CK(cudaEventRecord(s.done, ctx->stream));
        CK(cudaEventSynchronize(s.copied));
        ctx->carry_len = 0;
        ctx->next_slot = (si + 1) % NSLOT;
    }
    return TDG_OK;
}

// One array of a batch call: copied from `in` before the kernel, or to `out` after it
struct BatchPart {
    const void *in;
    void *out;
    size_t bytes;
};

// The batch calls (tdg_trim_batch, tdg_split_batch, tdg_match_batch) stage the reads' bytes, their
// offsets from the first read and `parts` in one device buffer the context keeps, each part 16-byte
// aligned.  launch(seqs, off, part) enqueues the kernel on those device addresses; then the output
// parts come back and the stream is synchronised.  Errors are reported as "<what>: ...".
template <class Launch>
int batch_run(tdg_ctx *ctx, const char *what, const char *seqs, const uint64_t *off, uint32_t n, std::initializer_list<BatchPart> parts,
              Launch launch)
{
    const size_t nbytes = (size_t)(off[n] - off[0]);
    std::vector<unsigned long long> rel(n + 1);
    for (uint32_t i = 0; i <= n; i++) rel[i] = off[i] - off[0];
    const size_t o_off = round_up(nbytes + 16, 16);
    size_t total = o_off + round_up((n + 1) * sizeof(uint64_t), 16);
    std::vector<size_t> at;
    for (const BatchPart &p : parts) {
        at.push_back(total);
        total += round_up(p.bytes, 16);
    }
    if (int rc = grow(ctx, ctx->batch, total, false)) return fail(ctx, rc, std::string(what) + ": " + ctx->err);
    uint8_t *d = (uint8_t *)ctx->batch.p;
    std::vector<uint8_t *> dev;
    for (size_t a : at) dev.push_back(d + a);
    const BatchPart *part = parts.begin();
    cudaError_t e = cudaSuccess;
    if (nbytes) e = cudaMemcpyAsync(d, seqs + off[0], nbytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + o_off, rel.data(), (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream);
    for (size_t k = 0; k < parts.size() && e == cudaSuccess; k++)
        if (part[k].in) e = cudaMemcpyAsync(dev[k], part[k].in, part[k].bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        launch(d, (const unsigned long long *)(d + o_off), dev.data());
        e = cudaGetLastError();
        ctx->launches += 1;
    }
    for (size_t k = 0; k < parts.size() && e == cudaSuccess; k++)
        if (part[k].out) e = cudaMemcpyAsync(part[k].out, dev[k], part[k].bytes, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(ctx, TDG_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
    if (e2 != cudaSuccess) return fail(ctx, TDG_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e2));
    return TDG_OK;
}

// The front tdg_split_block, tdg_split_count_block and tdg_split_count_device share: the block goes to
// sp_in (`kind` says whether `bytes` is host or device memory; either way sp_in carries the zero padding
// the kernels read past n), its line ends are found and split_records takes the decisions for its first
// `nrec` whole records (nrec = 0: there is none, and nothing ran past the line count).  prepare(nrec)
// grows the caller's own buffers and sets w.complex_flag before split_records is launched.  last_end
// (the terminator of the last record's last line) is valid once the caller has synchronised the stream.
template <class Prepare>
int split_front(tdg_ctx *ctx, const uint8_t *bytes, cudaMemcpyKind kind, size_t n, int final_block, uint64_t max_records,
                tdg::SplitWork &w, uint64_t &nrec, uint32_t &last_end, Prepare prepare)
{
    cudaStream_t st = ctx->stream;
    const uint32_t nbar = ctx->sp_nbar;
    int rc;
    nrec = 0;
    last_end = 0;

    // ---- the block, and its line ends
    const uint32_t n_tiles = (uint32_t)((n + tdg::SPLIT_TILE_BYTES - 1) / tdg::SPLIT_TILE_BYTES);
    if ((rc = grow(ctx, ctx->sp_in, round_up(n, 16) + 16, false))) return rc;
    if ((rc = grow(ctx, ctx->sp_tiles, (size_t)(n_tiles + 2) * sizeof(uint32_t), false))) return rc;
    CK(cudaMemcpyAsync(ctx->sp_in.p, bytes, n, kind, st));
    CK(cudaMemsetAsync((uint8_t *)ctx->sp_in.p + n, 0, round_up(n, 16) + 16 - n, st));
    memset(&w, 0, sizeof w);
    w.b.bytes = (const uint8_t *)ctx->sp_in.p;
    w.b.n = (uint32_t)n;
    w.b.final_block = final_block ? 1u : 0u;
    w.b.n_tiles = n_tiles;
    w.b.tile_count = (uint32_t *)ctx->sp_tiles.p;
    w.b.ends = nullptr;
    w.b.ends_cap = 0;
    tdg::lineend_count<<<n_tiles, 256, 0, st>>>(w.b);
    tdg::tile_scan<<<1, 1024, 0, st>>>(w.b.tile_count, n_tiles);
    ctx->launches += 2;
    uint32_t lines = 0;
    uint8_t last = 0;
    CK(cudaMemcpyAsync(&lines, w.b.tile_count + n_tiles, sizeof lines, cudaMemcpyDeviceToHost, st));
    if (kind == cudaMemcpyDeviceToDevice) CK(cudaMemcpyAsync(&last, (const uint8_t *)ctx->sp_in.p + n - 1, 1, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (kind == cudaMemcpyHostToDevice) last = bytes[n - 1];
    // the text after the last line end is a line of its own when the file ends here
    const bool open_tail = final_block && last != '\n' && last != '\r';
    const uint64_t total_lines = (uint64_t)lines + (open_tail ? 1 : 0);
    uint64_t records = total_lines / 4;
    if (records > max_records) records = max_records;
    if (records == 0) return TDG_OK;                 // the caller supplies more bytes (or stops at the end of the file)
    if ((rc = grow(ctx, ctx->sp_ends, (size_t)(total_lines + 1) * sizeof(uint32_t), false))) return rc;
    w.b.ends = (uint32_t *)ctx->sp_ends.p;
    w.b.ends_cap = lines;
    tdg::lineend_scatter<<<n_tiles, 256, 0, st>>>(w.b);
    ctx->launches += 1;
    if (open_tail) {
        const uint32_t end = (uint32_t)n;
        CK(cudaMemcpyAsync(w.b.ends + lines, &end, sizeof end, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpyAsync(&last_end, w.b.ends + (4 * records - 1), sizeof last_end, cudaMemcpyDeviceToHost, st));

    // ---- decisions
    if ((rc = grow(ctx, ctx->sp_rec, (size_t)records * sizeof(tdg::SplitRec), false))) return rc;
    if ((rc = grow(ctx, ctx->sp_flags, (size_t)records + 16, false))) return rc;
    if ((rc = prepare(records))) return rc;
    w.n_rec = (uint32_t)records;
    w.rec = (tdg::SplitRec *)ctx->sp_rec.p;
    w.flags = (uint8_t *)ctx->sp_flags.p;
    w.s.t = ctx->trim;
    w.s.bar = (const tdg::BarTable *)ctx->d_bar.p;
    w.bar_off = (const uint32_t *)ctx->sp_tabs.p;
    w.s.bar_len = w.bar_off + nbar + 1;
    w.barcodes = (const uint8_t *)(w.s.bar_len + nbar);
    w.s.cutlen = ctx->sp_cutlen;
    w.nbar = nbar;
    CK(cudaMemsetAsync(w.complex_flag, 0, sizeof(unsigned long long), st));
    tdg::split_records<<<(unsigned)((records + 7) / 8), 256, 0, st>>>(w);
    ctx->launches += 1;
    nrec = records;
    return TDG_OK;
}

// tdg_split_count_block / tdg_split_count_batch: every table they read is loaded and fits the matrix
int split_count_ready(tdg_ctx *ctx)
{
    if (!ctx->have_split_count || !ctx->have_split || !ctx->have_trim || !ctx->have_bar)
        return fail(ctx, TDG_ERR_STATE, "tdg_split_count_begin has not been called");
    if (!ctx->have_tags) return fail(ctx, TDG_ERR_STATE, "tdg_set_tags has not been called");
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "tdg_set_matrix / tdg_bind_matrix has not been called");
    if (ctx->max_col >= ctx->cols) return fail(ctx, TDG_ERR_ARG, "a tag column lies outside the matrix");
    if (ctx->sc_max_row >= ctx->rows) return fail(ctx, TDG_ERR_ARG, "a barcode row lies outside the matrix");
    return TDG_OK;
}

tdg::SplitCountArgs split_count_args(tdg_ctx *ctx)
{
    tdg::SplitCountArgs c;
    c.bar = (const tdg::BarTable *)ctx->sc_bar.p;
    c.tags = ctx->tags.t;
    c.tags.entries = (const tdg::TagEntry *)ctx->d_entries.p;
    c.tags.ext = (const uint64_t *)ctx->d_ext.p;
    c.row_of = (const int32_t *)ctx->sc_rows.p;
    c.matrix = ctx->d_matrix;
    c.cols = ctx->cols;
    return c;
}

#include "tdg_gzfeed.cuh"      // the host side of the device gzip feed (part of this unit)

}  // namespace

// ---------------------------------------------------------------------------

extern "C" {

int tdg_abi_version(void) { return TDG_ABI_VERSION; }

const char *tdg_last_error(const tdg_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int tdg_create(tdg_ctx **out, int device, size_t chunk_bytes)
{
    if (!out) return TDG_ERR_ARG;
    *out = nullptr;
    tdg_ctx *ctx = nullptr;   // CK reports into g_create_error while ctx is null
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, TDG_ERR_CUDA,
                    std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                        " (tagdigger_b200 has no CPU counting path)");
    if (device < 0 || device >= ndev) return fail(nullptr, TDG_ERR_ARG, "no such CUDA device");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, TDG_ERR_CUDA, std::string("device ") + prop.name + " is not sm_100 class; this library is built for sm_100a only");
    // dynamic shared memory a block may ask for: the opt-in limit minus the kernel's static part
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, tdg::count_kernel<true, false>));
    tdg_ctx *c = new (std::nothrow) tdg_ctx();
    if (!c) return fail(nullptr, TDG_ERR_NOMEM, "out of memory");
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin > fa.sharedSizeBytes ? prop.sharedMemPerBlockOptin - fa.sharedSizeBytes : 0;
    c->chunk_bytes = chunk_bytes ? chunk_bytes : ((size_t)64 << 20);
    if (const char *e = getenv("TDG_SEG_TILES")) c->force_seg_tiles = (uint32_t)atoi(e);
    if (const char *e = getenv("TDG_GENERAL")) c->force_general = atoi(e) != 0;
    if (c->chunk_bytes < 4096) c->chunk_bytes = 4096;
    std::string why;
    cudaError_t e2 = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e2 != cudaSuccess)
        why = cudaGetErrorString(e2);
    else if (grow_exact(c, c->d_state, 2 * sizeof(tdg::LineState), false) || grow_exact(c, c->d_totals, 4 * sizeof(unsigned long long), false))
        why = c->err;
    else if ((e2 = cudaMemset(c->d_state.p, 0, 2 * sizeof(tdg::LineState))) != cudaSuccess ||
             (e2 = cudaMemset(c->d_totals.p, 0, 4 * sizeof(unsigned long long))) != cudaSuccess)
        why = cudaGetErrorString(e2);
    if (!why.empty()) {
        tdg_destroy(c);
        return fail(nullptr, TDG_ERR_CUDA, "context set-up failed: " + why);
    }
    if (const char *e = getenv("TDG_FAIL_ALLOC")) c->fail_at = strtoull(e, nullptr, 10);
    *out = c;
    return TDG_OK;
}

void tdg_destroy(tdg_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    ctx->ahead.reset();          // the read-ahead thread writes into the pinned file buffers: joined before they are freed
    if (ctx->comm && tdg::nccl().CommDestroy) tdg::nccl().CommDestroy(ctx->comm);
    cudaStream_t stream = ctx->stream, copy_stream = ctx->copy_stream;
    delete ctx;                  // every buffer and event of the context
    if (stream) cudaStreamDestroy(stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
}

int tdg_set_tags(tdg_ctx *ctx, const char *bases, const uint64_t *off, const int32_t *col, uint32_t ntags,
                 uint32_t flags)
{
    if (!ctx || !off || !col || (!bases && off[ntags] != off[0])) return fail(ctx, TDG_ERR_ARG, "null argument");
    ctx->have_tags = false;
    std::string why = tdg::build_tag_table(bases, off, col, ntags, flags, ctx->tags);
    if (!why.empty()) return fail(ctx, TDG_ERR_ARG, "tdg_set_tags: " + why);
    ctx->max_col = 0;
    for (uint32_t i = 0; i < ntags; i++) {
        if (col[i] < 0) return fail(ctx, TDG_ERR_ARG, "tdg_set_tags: negative column");
        if ((uint32_t)col[i] > ctx->max_col) ctx->max_col = (uint32_t)col[i];
    }
    {
        CK(cudaSetDevice(ctx->device));
        CK(cudaStreamSynchronize(ctx->stream));
        size_t ne = ctx->tags.entries.size() * sizeof(tdg::TagEntry), nx = ctx->tags.ext.size() * sizeof(uint64_t);
        int rc;
        if ((rc = grow_exact(ctx, ctx->d_entries, ne, false)) || (rc = grow_exact(ctx, ctx->d_ext, std::max<size_t>(nx, 8), false))) return rc;
        if (ne) CK(cudaMemcpy(ctx->d_entries.p, ctx->tags.entries.data(), ne, cudaMemcpyHostToDevice));
        if (nx) CK(cudaMemcpy(ctx->d_ext.p, ctx->tags.ext.data(), nx, cudaMemcpyHostToDevice));
    }
    ctx->have_tags = true;
    return TDG_OK;
}

int tdg_set_matrix(tdg_ctx *ctx, uint32_t rows, uint32_t cols)
{
    if (!ctx || rows == 0 || cols == 0) return fail(ctx, TDG_ERR_ARG, "matrix must have at least one row and column");
    if ((uint64_t)rows * cols >= 0xFFFFFFFFull) return fail(ctx, TDG_ERR_ARG, "matrix must have fewer than 2^32 - 1 cells");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    int rc = grow_exact(ctx, ctx->matrix, (size_t)rows * cols * sizeof(int32_t), false);
    if (rc) return rc;
    ctx->d_matrix = (int32_t *)ctx->matrix.p;
    ctx->rows = rows;
    ctx->cols = cols;
    rc = size_replicas(ctx);
    if (rc) return rc;
    return tdg_zero_matrix(ctx);
}

int tdg_bind_matrix(tdg_ctx *ctx, void *dev_int32, uint32_t rows, uint32_t cols)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!dev_int32 || rows == 0 || cols == 0) return fail(ctx, TDG_ERR_ARG, "bad matrix");
    if ((uint64_t)rows * cols >= 0xFFFFFFFFull) return fail(ctx, TDG_ERR_ARG, "matrix must have fewer than 2^32 - 1 cells");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->matrix.reset();
    ctx->d_matrix = (int32_t *)dev_int32;
    ctx->rows = rows;
    ctx->cols = cols;
    return size_replicas(ctx);
}

int tdg_zero_matrix(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "no matrix");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->d_matrix, 0, (size_t)ctx->rows * ctx->cols * sizeof(int32_t), ctx->stream));
    return TDG_OK;
}

int tdg_begin_file(tdg_ctx *ctx, const char *bases, const uint32_t *off, const int32_t *row, const uint32_t *tag_off,
                   uint32_t npat, uint32_t flags)
{
    if (!ctx || !off || !row || !tag_off) return fail(ctx, TDG_ERR_ARG, "null argument");
    if (ctx->carry_len) return fail(ctx, TDG_ERR_STATE, "previous file was not ended (tdg_end_file)");
    ctx->have_bar = false;
    std::string why = tdg::build_bar_table(bases, off, row, tag_off, npat, flags, ctx->bar_blob);
    if (!why.empty()) return fail(ctx, TDG_ERR_ARG, "tdg_begin_file: " + why);
    ctx->max_row = 0;
    for (uint32_t i = 0; i < npat; i++) {
        if (row[i] < 0) return fail(ctx, TDG_ERR_ARG, "tdg_begin_file: negative row");
        if ((uint32_t)row[i] > ctx->max_row) ctx->max_row = (uint32_t)row[i];
    }
    {
        CK(cudaSetDevice(ctx->device));
        // the previous file's kernels read the old table
        CK(cudaStreamSynchronize(ctx->stream));
        int rc = grow_exact(ctx, ctx->d_bar, round_up(ctx->bar_blob.size(), 16), false);
        if (rc) return rc;
        CK(cudaMemcpy(ctx->d_bar.p, ctx->bar_blob.data(), ctx->bar_blob.size(), cudaMemcpyHostToDevice));
        CK(cudaMemsetAsync(ctx->d_state.p, 0, 2 * sizeof(tdg::LineState), ctx->stream));
        CK(cudaMemsetAsync(ctx->d_totals.p, 0, 4 * sizeof(unsigned long long), ctx->stream));
        ctx->state_cur = 0;
    }
    ctx->have_bar = true;
    ctx->file_open = true;
    return TDG_OK;
}

int tdg_reset_file(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_bar) return fail(ctx, TDG_ERR_STATE, "tdg_begin_file has not been called");
    if (ctx->carry_len) return fail(ctx, TDG_ERR_STATE, "previous file was not ended (tdg_end_file)");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->d_state.p, 0, 2 * sizeof(tdg::LineState), ctx->stream));
    CK(cudaMemsetAsync(ctx->d_totals.p, 0, 4 * sizeof(unsigned long long), ctx->stream));
    ctx->state_cur = 0;
    return TDG_OK;
}

int tdg_submit(tdg_ctx *ctx, const void *bytes, size_t n, uint64_t reads_limit)
{
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (n == 0) return TDG_OK;
    if (!bytes) return fail(ctx, TDG_ERR_ARG, "null buffer");
    CK(cudaSetDevice(ctx->device));
    rc = submit_impl(ctx, (const uint8_t *)bytes, n, reads_limit, true);
    if (rc) ctx->carry_len = 0;          // the file is given up, as in tdg_count_file: tdg_begin_file starts the next one
    return rc;
}

int tdg_end_file(tdg_ctx *ctx, uint64_t reads_limit)
{
    int rc = need_ready(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ensure_slots(ctx);
    if (rc == TDG_OK) rc = end_file_impl(ctx, reads_limit);
    if (rc) ctx->carry_len = 0;
    return rc;
}

int tdg_count_device(tdg_ctx *ctx, const void *dev_bytes, size_t n, uint64_t line_base, int prev_kind,
                     uint64_t reads_limit)
{
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (n && !dev_bytes) return fail(ctx, TDG_ERR_ARG, "null buffer");
    if (line_base != TDG_LINE_CHAINED && (prev_kind < 0 || prev_kind > 3)) return fail(ctx, TDG_ERR_ARG, "bad prev_kind");
    CK(cudaSetDevice(ctx->device));
    return launch_chunk<true>(ctx, dev_bytes, n, line_base, prev_kind, reads_limit);
}

int tdg_count_lines_device(tdg_ctx *ctx, const void *dev_bytes, size_t n, uint64_t line_base, int prev_kind,
                           uint64_t state[2])
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!state || (n && !dev_bytes)) return fail(ctx, TDG_ERR_ARG, "null argument");
    if (prev_kind < 0 || prev_kind > 3) return fail(ctx, TDG_ERR_ARG, "bad prev_kind");
    CK(cudaSetDevice(ctx->device));
    if (n == 0) {
        state[0] = line_base;
        state[1] = (uint64_t)prev_kind;
        return TDG_OK;
    }
    rc = launch_chunk<false>(ctx, dev_bytes, n, line_base, prev_kind, 0);
    if (rc) return rc;
    tdg::LineState st;
    CK(cudaMemcpyAsync(&st, (tdg::LineState *)ctx->d_state.p + ctx->state_cur, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    state[0] = st.next_line;
    state[1] = st.prev_kind;
    return TDG_OK;
}

int tdg_sync(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->copy_stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TDG_OK;
}

int tdg_file_totals(tdg_ctx *ctx, uint64_t totals[4])
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!totals) return fail(ctx, TDG_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    unsigned long long t[4];
    tdg::LineState st;
    CK(cudaMemcpyAsync(t, ctx->d_totals.p, sizeof(t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&st, (tdg::LineState *)ctx->d_state.p + ctx->state_cur, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    totals[0] = t[0];
    totals[1] = t[1];
    totals[2] = t[2];
    totals[3] = st.next_line;
    return TDG_OK;
}

int tdg_read_matrix(tdg_ctx *ctx, int32_t *out)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "no matrix");
    CK(cudaSetDevice(ctx->device));
    if (out)
        CK(cudaMemcpyAsync(out, ctx->d_matrix, (size_t)ctx->rows * ctx->cols * sizeof(int32_t), cudaMemcpyDeviceToHost,
                           ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TDG_OK;
}

int tdg_matrix_min(tdg_ctx *ctx, int32_t *out)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "no matrix");
    if (!out) return fail(ctx, TDG_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    int32_t *d_min = (int32_t *)((unsigned long long *)ctx->d_totals.p + 3);          // the spare word behind the three totals
    const int32_t init = 0x7FFFFFFF;
    CK(cudaMemcpyAsync(d_min, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t cells = ctx->rows * ctx->cols;
    unsigned grid = (unsigned)std::min<size_t>(((size_t)cells + 255) / 256, (size_t)ctx->sm_count * 8);
    tdg::min_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_matrix, cells, d_min);
    CK(cudaGetLastError());
    ctx->launches += 1;
    CK(cudaMemcpyAsync(out, d_min, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TDG_OK;
}

void *tdg_matrix_device_ptr(tdg_ctx *ctx) { return ctx ? ctx->d_matrix : nullptr; }
void *tdg_stream(tdg_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int tdg_stream_wait(tdg_ctx *ctx, void *other_stream)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    if ((rc = make_event(ctx, ctx->handoff))) return rc;
    CK(cudaEventRecord(ctx->handoff, (cudaStream_t)other_stream));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->handoff, 0));
    return TDG_OK;
}

int tdg_other_stream_wait(tdg_ctx *ctx, void *other_stream)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    if ((rc = make_event(ctx, ctx->handoff))) return rc;
    CK(cudaEventRecord(ctx->handoff, ctx->stream));
    CK(cudaStreamWaitEvent((cudaStream_t)other_stream, ctx->handoff, 0));
    return TDG_OK;
}

// ---------------------------------------------------------------------------
// Multi-GPU: one process (or thread) per GPU, one context each; the only exchange of the path is
// the sum of the count matrices.

int tdg_comm_unique_id(void *out128)
{
    if (!out128) return fail(nullptr, TDG_ERR_ARG, "null argument");
    tdg::NcclApi &N = tdg::nccl();
    if (!N.load()) return fail(nullptr, TDG_ERR_STATE, N.why);
    tdg::NcclApi::UniqueId id;
    int rc = N.GetUniqueId(&id);
    if (rc) return fail(nullptr, TDG_ERR_CUDA, "ncclGetUniqueId: " + N.message(rc));
    memcpy(out128, &id, sizeof(id));
    return TDG_OK;
}

int tdg_comm_init(tdg_ctx *ctx, const void *id128, int nranks, int rank)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, TDG_ERR_ARG, "bad communicator arguments");
    tdg::NcclApi &N = tdg::nccl();
    if (!N.load()) return fail(ctx, TDG_ERR_STATE, N.why);
    CK(cudaSetDevice(ctx->device));
    if (ctx->comm) { N.CommDestroy(ctx->comm); ctx->comm = nullptr; }
    tdg::NcclApi::UniqueId id;
    memcpy(&id, id128, sizeof(id));
    int nrc = N.CommInitRank(&ctx->comm, nranks, id, rank);
    if (nrc) { ctx->comm = nullptr; return fail(ctx, TDG_ERR_CUDA, "ncclCommInitRank: " + N.message(nrc)); }
    ctx->comm_ranks = nranks;
    return TDG_OK;
}

int tdg_allreduce_matrix(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "no matrix");
    if (!ctx->comm) return ctx->comm_ranks == 1 ? TDG_OK : fail(ctx, TDG_ERR_STATE, "tdg_comm_init has not been called");
    CK(cudaSetDevice(ctx->device));
    tdg::NcclApi &N = tdg::nccl();
    int nrc = N.AllReduce(ctx->d_matrix, ctx->d_matrix, (size_t)ctx->rows * ctx->cols, tdg::NcclApi::kInt32, tdg::NcclApi::kSum,
                          ctx->comm, ctx->stream);
    if (nrc) return fail(ctx, TDG_ERR_CUDA, "ncclAllReduce: " + N.message(nrc));
    return TDG_OK;
}

int tdg_finish(tdg_ctx *ctx, int32_t *out, uint64_t totals[4])
{
    int rc = tdg_allreduce_matrix(ctx);
    if (rc) return rc;
    if (totals) {
        rc = tdg_file_totals(ctx, totals);
        if (rc) return rc;
    }
    return tdg_read_matrix(ctx, out);
}

void *tdg_host_alloc(tdg_ctx *ctx, size_t n)
{
    if (!ctx) return nullptr;
    void *p = nullptr;
    cudaSetDevice(ctx->device);
    if (cudaHostAlloc(&p, n ? n : 1, cudaHostAllocDefault) != cudaSuccess) {
        ctx->err = "cudaHostAlloc failed";
        return nullptr;
    }
    return p;
}
void tdg_host_free(tdg_ctx *ctx, void *p)
{
    (void)ctx;
    if (p) cudaFreeHost(p);
}
void *tdg_device_alloc(tdg_ctx *ctx, size_t n)
{
    if (!ctx) return nullptr;
    void *p = nullptr;
    cudaSetDevice(ctx->device);
    if (cudaMalloc(&p, n ? n : 1) != cudaSuccess) {
        ctx->err = "cudaMalloc failed";
        return nullptr;
    }
    return p;
}
void tdg_device_free(tdg_ctx *ctx, void *p)
{
    if (!ctx || !p) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(p);
}
int tdg_memcpy_h2d(tdg_ctx *ctx, void *dev, const void *host, size_t n)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dev, host, n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TDG_OK;
}
int tdg_memcpy_d2h(tdg_ctx *ctx, void *host, const void *dev, size_t n)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(host, dev, n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TDG_OK;
}

uint64_t tdg_launch_count(const tdg_ctx *ctx) { return ctx ? ctx->launches : 0; }

int tdg_timing_begin(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    ctx->tev.resize(2 * MAX_TIMED);      // (created as they are first used: timed_start)
    ctx->tev_used = 0;
    ctx->timing = true;
    return TDG_OK;
}

int tdg_timing_end(tdg_ctx *ctx, double *kernel_ms, uint32_t *nlaunch)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    double ms = 0;
    for (int i = 0; i + 1 < ctx->tev_used; i += 2) {
        float t = 0;
        CK(cudaEventElapsedTime(&t, ctx->tev[i], ctx->tev[i + 1]));
        ms += t;
    }
    if (kernel_ms) *kernel_ms = ms;
    if (nlaunch) *nlaunch = (uint32_t)(ctx->tev_used / 2);
    ctx->timing = false;
    return TDG_OK;
}

// ---------------------------------------------------------------------------
// Whole-file streaming: a reader thread (read() or zlib inflate) fills pinned
// buffers; the calling thread feeds them to the GPU.

namespace {

int ensure_file_bufs(tdg_ctx *ctx, int set)
{
    for (Buf &b : ctx->file_buf[set]) {
        int rc = grow_exact(ctx, b, ctx->chunk_bytes, true);
        if (rc) return rc;
    }
    return TDG_OK;
}

size_t file_chunk(const tdg_ctx *ctx, uint64_t reads_limit)
{
    // With a read limit the reference stops reading at the maxreads'th sequence line
    // (tagdigger_fun.py:272-273): feed smaller pieces, so that little is read, inflated and copied
    // beyond that point.
    const bool small = reads_limit < ((uint64_t)1 << 60) && 4 * reads_limit <= ctx->chunk_bytes + 2;       // the limit's line can lie in the first piece
    return small ? std::min<size_t>(ctx->chunk_bytes, (size_t)8 << 20) : ctx->chunk_bytes;
}

std::unique_ptr<FileReader> start_reader(tdg_ctx *ctx, const char *path, bool gz, size_t chunk, int set, const GzHandover *ho)
{
    std::unique_ptr<FileReader> r(new FileReader());
    for (int i = 0; i < FileReader::NBUF; i++) r->bufs[i].p = (uint8_t *)ctx->file_buf[set][i].p;
    r->path = path;
    r->gz = gz;
    r->chunk = chunk;
    r->set = set;
    if (ho) r->ho = *ho;
    r->start();
    return r;
}

}  // namespace

int tdg_count_file2(tdg_ctx *ctx, const char *path, int gz, uint64_t reads_limit, uint64_t totals[4], const char *next_path, int next_gz)
{
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!path) return fail(ctx, TDG_ERR_ARG, "null path");
    CK(cudaSetDevice(ctx->device));
    rc = ensure_slots(ctx);
    if (rc) return rc;
    const size_t chunk = file_chunk(ctx, reads_limit);
    LimitState lim;
    lim.init(reads_limit, ctx->chunk_bytes);

    ctx->last_file[0] = ctx->last_file[1] = 0;
    ctx->last_file[2] = -1;
    // a reader that was started for this file while the one before it was counted
    std::unique_ptr<FileReader> reader;
    if (ctx->ahead && ctx->ahead->path == path && ctx->ahead->gz == (gz != 0) && ctx->ahead->chunk == chunk) reader = std::move(ctx->ahead);
    ctx->ahead.reset();
    const int set = reader ? reader->set : 0;
    rc = ensure_file_bufs(ctx, set);
    if (rc) return rc;
    // ... and the one for the file that comes next (files the device gzip feed takes are not read ahead)
    if (next_path && *next_path && std::string(next_path) != path && !(next_gz && gz_device_wanted(ctx, next_path, reads_limit))) {
        struct stat sb;
        if (stat(next_path, &sb) == 0 && S_ISREG(sb.st_mode)) {
            rc = ensure_file_bufs(ctx, set ^ 1);
            if (rc) return rc;
            ctx->ahead = start_reader(ctx, next_path, next_gz != 0, chunk, set ^ 1, nullptr);
        }
    }

    // Ordinary gzip files are inflated on the DEVICE (tdg_gzdev.cuh): the compressed bytes cross
    // PCIe, the text is born in HBM.  Whatever that feed does not take -- small files, a read
    // limit, and the rest of any stream with something unusual in it -- goes through the host
    // feeder below, which resumes exactly where the device feed stopped.
    tdg::Utf8State u8;
    GzHandover ho;
    int result = TDG_OK;
    bool at_eof = false;
    if (!reader && gz && gz_device_wanted(ctx, path, reads_limit)) {
        bool handled = false;
        size_t dcarry = 0;
        GzCountSink sink(reads_limit, &lim);
        GzStats gst;
        result = gz_device_feed(ctx, path, sink, handled, ho, dcarry, gst, &u8);
        ctx->last_file[0] = gst.rounds;
        ctx->last_file[1] = gst.accepted;
        ctx->last_file[2] = !handled ? -1 : (ho.active ? 1 : 0);
        if (result == TDG_OK && handled && dcarry) {
            // the bytes behind the last line end become the host path's carry
            Slot &cs = ctx->slot[ctx->next_slot];
            result = grow_carry(ctx, cs.carry, dcarry, 0);
            if (result == TDG_OK) {
                CK(cudaMemcpyAsync(cs.carry.p, ctx->gz_text.p, dcarry, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
                ctx->carry_len = dcarry;
                lim.last_byte = ((const uint8_t *)cs.carry.p)[dcarry - 1];
                if (lim.careful) lim.ll.prev_cr = lim.last_byte == '\r';
            }
        }
        at_eof = handled && !ho.active;                      // the whole file went through the device
    }
    // the host feeder: from the start, or where the device feed handed over (none when that feed took the whole file or failed)
    if (!reader && result == TDG_OK && !at_eof) reader = start_reader(ctx, path, gz != 0, chunk, set, ho.active ? &ho : nullptr);

    const bool fdebug = getenv("TDG_FILE_DEBUG") != nullptr;
    const auto ft0 = std::chrono::steady_clock::now();
    double ms_wait = 0, ms_submit = 0;
    int bi = 0;
    // the read with index maxreads-1 is line 4*maxreads-3: everything up to line end number
    // 4*maxreads-2 is needed, nothing beyond it is looked at (LimitState)
    while (reader) {
        FileReader &fr = *reader;
        FileReader::Buf &b = fr.bufs[bi];
        const auto fw0 = std::chrono::steady_clock::now();
        {
            std::unique_lock<std::mutex> lk(fr.mu);
            fr.cv.wait(lk, [&] { return b.state == 1; });
        }
        const auto fw1 = std::chrono::steady_clock::now();
        ms_wait += std::chrono::duration<double, std::milli>(fw1 - fw0).count();
        if (b.err) { result = fail(ctx, b.err, b.msg); break; }
        if (b.n == 0) { at_eof = true; break; }
        size_t use = b.n;
        {
            const int go = limit_admits(ctx, lim, b.n);
            if (go < 0) { result = go; break; }
            if (go == 0) use = lim.ll.feed(b.p, b.n);
            if (use) lim.last_byte = b.p[use - 1];
        }
        // text mode: the bytes the loop reads must be valid UTF-8 (open(f, 'r'), errors='strict')
        if (b.high || u8.need) {
            long long bad = tdg::utf8_feed(u8, b.p, use);
            if (bad >= 0) {
                result = fail(ctx, TDG_ERR_UTF8, "position " + std::to_string(bad) + ": invalid UTF-8 in " + path);
                break;
            }
        } else {
            u8.offset += use;
        }
        if (use) result = submit_impl(ctx, b.p, use, reads_limit, true);
        ms_submit += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - fw1).count();
        {
            std::lock_guard<std::mutex> lk(fr.mu);
            b.state = 0;
        }
        fr.cv.notify_all();
        if (result || lim.ll.reached) break;
        bi = (bi + 1) % FileReader::NBUF;
    }
    reader.reset();                                          // stops and joins the reading thread
    if (result == TDG_OK && at_eof && tdg::utf8_finish(u8) >= 0)
        result = fail(ctx, TDG_ERR_UTF8, "position " + std::to_string(tdg::utf8_finish(u8)) + ": unexpected end of data in " + path);
    if (result == TDG_OK) result = end_file_impl(ctx, reads_limit);
    if (result != TDG_OK) ctx->carry_len = 0;
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->stream);
    if (result == TDG_OK && totals) result = tdg_file_totals(ctx, totals);
    if (fdebug)
        fprintf(stderr, "tdg_count_file %s: %.2f ms (waiting for the reader %.2f, validate + submit %.2f, end of file + totals %.2f)\n", path,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - ft0).count(), ms_wait, ms_submit,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - ft0).count() - ms_wait - ms_submit);
    return result;
}

int tdg_count_file(tdg_ctx *ctx, const char *path, int gz, uint64_t reads_limit, uint64_t totals[4])
{
    return tdg_count_file2(ctx, path, gz, reads_limit, totals, nullptr, 0);
}

// How the last tdg_count_file fed its file: info[0] rounds of the device gzip feed, [1] chunks (or BGZF
// members) they accepted, [2] 0 = the whole file went through the device, 1 = the host feeder took over
// somewhere, -1 = host feeder only.
int tdg_last_file_info(tdg_ctx *ctx, int64_t info[3])
{
    if (!ctx || !info) return fail(ctx, TDG_ERR_ARG, "null argument");
    for (int i = 0; i < 3; i++) info[i] = ctx->last_file[i];
    return TDG_OK;
}

// Gives the working buffers of the device-side gzip feed back (a 1.2 GB round holds about 12 GB:
// tokens, symbols, windows, text), and the staging buffer of the batch calls.  They are kept between
// calls otherwise.
int tdg_release_scratch(tdg_ctx *ctx)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaStreamSynchronize(ctx->copy_stream));
    // gz_tabs stays: gz_tables uploads the tables once per context.  The pinned gz_h* buffers stay too:
    // they are small (a round's chunk metadata and CRCs, the tail of its text searched for a line end).
    for (Buf *b : {&ctx->gz_comp, &ctx->gz_comp2, &ctx->gz_syms, &ctx->gz_sym2, &ctx->gz_ntok, &ctx->gz_meta, &ctx->gz_cand, &ctx->gz_ncand,
                   &ctx->gz_windows, &ctx->gz_text, &ctx->gz_crc, &ctx->gz_lens, &ctx->gz_offs, &ctx->gz_carry, &ctx->gz_cold, &ctx->batch})
        b->reset();
    return TDG_OK;
}

// The device-side gzip feed by itself: inflates `path` into dst (host memory) the way
// tdg_count_file does -- rounds on the device, the rest, if any, through the host feeder -- and
// reports what happened.  info[0] rounds, [1] chunks, [2] chunks accepted, [3] 0 all on the device /
// 1 host reader resumed / 2 zlib / -1 not taken by the device feed at all; ms[0..5]: upload, scan,
// decode, windows + resolve, CRC fold / UTF-8, sink.
int tdg_gz_inflate_host(tdg_ctx *ctx, const char *path, void *dst, size_t cap, uint64_t *n_out, int64_t info[4], double ms[6])
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!path || !dst || !n_out) return fail(ctx, TDG_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    rc = ensure_slots(ctx);
    if (rc) return rc;
    ctx->ahead.reset();
    rc = ensure_file_bufs(ctx, 0);
    if (rc) return rc;
    GzCopySink sink((uint8_t *)dst, cap);
    GzHandover ho;
    GzStats st;
    bool handled = false;
    size_t carry = 0;
    rc = gz_device_feed(ctx, path, sink, handled, ho, carry, st, nullptr);
    if (rc) return rc;
    if (info) {
        info[0] = st.rounds;
        info[1] = st.chunks;
        info[2] = st.accepted;
        info[3] = !handled ? -1 : (!ho.active ? 0 : (ho.to_zlib ? 2 : 1));
    }
    if (ms) {
        ms[0] = st.ms_upload;
        ms[1] = st.ms_scan;
        ms[2] = st.ms_decode;
        ms[3] = st.ms_resolve;
        ms[4] = st.ms_host;
        ms[5] = st.ms_sink;
    }
    size_t used = sink.used;
    if (!handled || ho.active) {
        tdg::Feeder feed;
        int orc = open_feed(feed, path, true, &ho);
        if (orc) return fail(ctx, orc, feed.error());
        for (;;) {
            if (used == cap) return fail(ctx, TDG_ERR_ARG, "output buffer too small");
            long long r = feed.fill((uint8_t *)dst + used, std::min<size_t>(cap - used, (size_t)64 << 20));
            if (r < 0) {
                *n_out = used;
                return fail(ctx, (int)r, feed.error());
            }
            if (r == 0) break;
            used += (size_t)r;
        }
    }
    *n_out = used;
    return TDG_OK;
}

// The member chain of a BGZF file, walked on the host with the feeder's header parser (no context: errors go
// to tdg_last_error(NULL)).  *n receives the number of members; off / isize receive them when cap holds them.
int tdg_bgzf_index(const char *path, uint64_t *off, uint32_t *isize, size_t cap, size_t *n)
{
    if (!path || !n || (cap && (!off || !isize))) return fail(nullptr, TDG_ERR_ARG, "null argument");
    GzMap map;
    if (!gz_map_file(map, path)) return fail(nullptr, TDG_ERR_IO, std::string("cannot open ") + path);
    std::vector<uint64_t> o;
    std::vector<uint32_t> s;
    const std::string why = bgzf_chain(map, o, s);
    if (!why.empty()) return fail(nullptr, TDG_ERR_GZIP, std::string(path) + " is not a BGZF member chain: " + why);
    *n = o.size();
    if (!cap) return TDG_OK;
    if (cap < o.size()) return fail(nullptr, TDG_ERR_ARG, "tdg_bgzf_index: room for " + std::to_string(cap) + " members, the file has " +
                                                                std::to_string(o.size()));
    memcpy(off, o.data(), o.size() * 8);
    memcpy(isize, s.data(), s.size() * 4);
    return TDG_OK;
}

// The BGZF members in [c_lo, c_hi) of `path`, inflated on the device into caller device memory (gz_bgzf_inflate_range).
int tdg_bgzf_inflate_device(tdg_ctx *ctx, const char *path, uint64_t c_lo, uint64_t c_hi, void *dst, size_t cap, uint64_t *n, int *high)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!path || !n || !high || (!dst && cap)) return fail(ctx, TDG_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    rc = ensure_slots(ctx);
    if (rc) return rc;
    ctx->ahead.reset();                      // the read-ahead thread writes into the pinned file buffers the upload uses
    rc = ensure_file_bufs(ctx, 0);
    if (rc) return rc;
    uint64_t got = 0;
    bool hi = false;
    rc = gz_bgzf_inflate_range(ctx, path, (size_t)c_lo, (size_t)c_hi, (uint8_t *)dst, cap, got, hi);
    if (rc) return rc;
    *n = got;
    *high = hi ? 1 : 0;
    return TDG_OK;
}

// ---------------------------------------------------------------------------
// Trim decision (barcode splitter), csrc/tdg_trim.cuh

int tdg_set_trim(tdg_ctx *ctx, const char *site0, const char *site1, const char *a0, uint32_t nbar, const char *a1,
                 const uint32_t *a1_off, const uint32_t *cand_off, const uint16_t *cand_len, const int16_t *cand_idx,
                 const uint8_t *cand_which)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!site0 || !site1 || !a0 || !a1 || !a1_off || !cand_off || (cand_off[nbar] && (!cand_len || !cand_idx || !cand_which)))
        return fail(ctx, TDG_ERR_ARG, "null argument");
    ctx->have_trim = false;
    const size_t l0 = strlen(site0), l1 = strlen(site1), la0 = strlen(a0);
    if (l0 == 0 || l1 == 0) return fail(ctx, TDG_ERR_ARG, "tdg_set_trim: restriction sites must not be empty");
    const uint32_t ncand = cand_off[nbar];
    std::vector<tdg::TrimCand> cand(ncand);
    for (uint32_t b = 0; b < nbar; b++) {
        if (a1_off[b + 1] < a1_off[b] || cand_off[b + 1] < cand_off[b]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
        for (uint32_t c = cand_off[b]; c < cand_off[b + 1]; c++) {
            size_t have = cand_which[c] ? (size_t)(a1_off[b + 1] - a1_off[b]) : la0;
            if (cand_len[c] == 0 || cand_len[c] > have)
                return fail(ctx, TDG_ERR_ARG, "tdg_set_trim: candidate " + std::to_string(c) + " is longer than its adapter string");
            cand[c].len = cand_len[c];
            cand[c].idx = cand_idx[c];
            cand[c].which = cand_which[c] ? 1u : 0u;
        }
    }
    // blob: site0 | site1 | a0 | a1 | a1_off | cand_off | cand   (each part 16-byte aligned)
    size_t o_site0 = 0, o_site1 = round_up(o_site0 + l0, 16), o_a0 = round_up(o_site1 + l1, 16),
           o_a1 = round_up(o_a0 + la0, 16), o_a1off = round_up(o_a1 + a1_off[nbar], 16),
           o_coff = round_up(o_a1off + (nbar + 1) * sizeof(uint32_t), 16),
           o_cand = round_up(o_coff + (nbar + 1) * sizeof(uint32_t), 16),
           total = round_up(o_cand + ncand * sizeof(tdg::TrimCand), 16) + 16;
    std::vector<uint8_t> blob(total, 0);
    memcpy(blob.data() + o_site0, site0, l0);
    memcpy(blob.data() + o_site1, site1, l1);
    memcpy(blob.data() + o_a0, a0, la0);
    if (a1_off[nbar]) memcpy(blob.data() + o_a1, a1, a1_off[nbar]);
    memcpy(blob.data() + o_a1off, a1_off, (nbar + 1) * sizeof(uint32_t));
    memcpy(blob.data() + o_coff, cand_off, (nbar + 1) * sizeof(uint32_t));
    if (ncand) memcpy(blob.data() + o_cand, cand.data(), ncand * sizeof(tdg::TrimCand));
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    rc = grow_exact(ctx, ctx->d_trim, total, false);
    if (rc) return rc;
    const uint8_t *d = (const uint8_t *)ctx->d_trim.p;
    CK(cudaMemcpy(ctx->d_trim.p, blob.data(), total, cudaMemcpyHostToDevice));
    tdg::TrimArgs &t = ctx->trim;
    memset(&t, 0, sizeof(t));
    t.site0 = d + o_site0;
    t.site1 = d + o_site1;
    t.len0 = (uint32_t)l0;
    t.len1 = (uint32_t)l1;
    t.a0 = d + o_a0;
    t.a1 = d + o_a1;
    t.a1_off = (const uint32_t *)(d + o_a1off);
    t.cand_off = (const uint32_t *)(d + o_coff);
    t.cand = (const tdg::TrimCand *)(d + o_cand);
    ctx->trim_nbar = nbar;
    ctx->have_trim = true;
    return TDG_OK;
}

int tdg_trim_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, const int32_t *bar, const uint32_t *start,
                   uint32_t n, int32_t *slice2)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_trim) return fail(ctx, TDG_ERR_STATE, "tdg_set_trim has not been called");
    if (n == 0) return TDG_OK;
    if (!off || !bar || !start || !slice2 || (!seqs && off[n] != off[0])) return fail(ctx, TDG_ERR_ARG, "null argument");
    for (uint32_t i = 0; i < n; i++) {
        if (bar[i] < 0 || (uint32_t)bar[i] >= ctx->trim_nbar) return fail(ctx, TDG_ERR_ARG, "barcode index out of range");
        if (off[i + 1] < off[i]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
    }
    CK(cudaSetDevice(ctx->device));
    return batch_run(ctx, "tdg_trim_batch", seqs, off, n, {{bar, nullptr, n * sizeof(int32_t)}, {start, nullptr, n * sizeof(uint32_t)}, {nullptr, slice2, n * sizeof(int32_t)}},
                     [&](const uint8_t *d, const unsigned long long *d_off, uint8_t *const *part) {
                         tdg::TrimArgs t = ctx->trim;
                         t.seqs = d;
                         t.off = d_off;
                         t.bar = (const int32_t *)part[0];
                         t.start = (const uint32_t *)part[1];
                         t.n = n;
                         t.out = (int32_t *)part[2];
                         const unsigned per = tdg::TRIM_THREADS / 32;
                         tdg::trim_kernel<<<(n + per - 1) / per, tdg::TRIM_THREADS, 0, ctx->stream>>>(t);
                     });
}

int tdg_split_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, uint32_t n, const uint32_t *bar_len,
                    uint32_t nbar, uint32_t cutlen, int32_t *bar_out, int32_t *slice2)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_trim) return fail(ctx, TDG_ERR_STATE, "tdg_set_trim has not been called");
    if (!ctx->have_bar) return fail(ctx, TDG_ERR_STATE, "tdg_begin_file has not been called");
    if (nbar != ctx->trim_nbar || ctx->max_row >= nbar)
        return fail(ctx, TDG_ERR_ARG, "barcode table, trim tables and bar_len disagree on the number of barcodes");
    if (n == 0) return TDG_OK;
    if (!off || !bar_len || !bar_out || !slice2 || (!seqs && off[n] != off[0])) return fail(ctx, TDG_ERR_ARG, "null argument");
    for (uint32_t i = 0; i < n; i++)
        if (off[i + 1] < off[i]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
    CK(cudaSetDevice(ctx->device));
    return batch_run(ctx, "tdg_split_batch", seqs, off, n,
                     {{bar_len, nullptr, nbar * sizeof(uint32_t)}, {nullptr, bar_out, n * sizeof(int32_t)}, {nullptr, slice2, n * sizeof(int32_t)}},
                     [&](const uint8_t *d, const unsigned long long *d_off, uint8_t *const *part) {
                         tdg::SplitArgs a;
                         a.t = ctx->trim;
                         a.t.seqs = d;
                         a.t.off = d_off;
                         a.t.n = n;
                         a.t.out = (int32_t *)part[2];
                         a.bar = (const tdg::BarTable *)ctx->d_bar.p;
                         a.bar_len = (const uint32_t *)part[0];
                         a.cutlen = cutlen;
                         a.bar_out = (int32_t *)part[1];
                         const unsigned per = tdg::TRIM_THREADS / 32;
                         tdg::split_kernel<<<(n + per - 1) / per, tdg::TRIM_THREADS, 0, ctx->stream>>>(a);
                     });
}

// ---------------------------------------------------------------------------
// Streaming barcode splitter, csrc/tdg_split.cuh

// BGZF members of the splitter's streams (tdg_bgzf.cuh).  Barcode b's stream gains the device bytes
// d_new[off[b] .. off[b+1]) behind its pending tail; every complete 65,280 bytes become a member and the
// rest is the new tail.  finish: the tails become the last members, and every file gets the EOF member.
// Members are planned here, one CTA each deflates them, and they come back end to end in barcode order:
// *out (pinned, owned by the context) with barcode b's bytes at [(*out_off)[b], (*out_off)[b+1]).
static int bgzf_run(tdg_ctx *ctx, const uint8_t *d_new, const uint64_t *off, bool finish, const uint8_t **out,
                    const uint64_t **out_off)
{
    namespace bz = tdg::bz;
    const uint32_t nbar = ctx->sp_nbar;
    cudaStream_t st = ctx->stream;
    uint8_t *tails = (uint8_t *)ctx->bz_tail.p;
    std::vector<bz::Member> mem;
    std::vector<bz::Copy> cp;
    std::vector<uint32_t> first(nbar + 1);
    uint64_t in_total = 0, slot_total = 0;
    auto add = [&](const uint8_t *s0, uint32_t l0, const uint8_t *s1, uint32_t l1) {
        bz::Member m;
        m.src0 = s0;
        m.len0 = l0;
        m.src1 = s1;
        m.len1 = l1;
        m.in_off = in_total;
        m.slot = slot_total;
        in_total += l0 + l1;
        slot_total += round_up(l0 + l1 + bz::SLOT_EXTRA, 16);
        mem.push_back(m);
    };
    for (uint32_t b = 0; b < nbar; b++) {
        first[b] = (uint32_t)mem.size();
        uint8_t *tail = tails + (size_t)b * bz::BLOCK;
        const uint32_t t = ctx->bz_tail_len[b];
        if (finish) {
            if (t) add(tail, t, nullptr, 0);
            add(nullptr, 0, nullptr, 0);                 // the end-of-file member
            ctx->bz_tail_len[b] = 0;
            continue;
        }
        const uint64_t L = off[b + 1] - off[b];
        const uint8_t *src = d_new + off[b];
        if (t + L < bz::BLOCK) {
            if (L) cp.push_back(bz::Copy{src, tail + t, L});
            ctx->bz_tail_len[b] = (uint32_t)(t + L);
            continue;
        }
        add(tail, t, src, bz::BLOCK - t);
        uint64_t p = bz::BLOCK - t;
        for (; p + bz::BLOCK <= L; p += bz::BLOCK) add(nullptr, 0, src + p, bz::BLOCK);
        if (p < L) cp.push_back(bz::Copy{src + p, tail, L - p});
        ctx->bz_tail_len[b] = (uint32_t)(L - p);
    }
    first[nbar] = (uint32_t)mem.size();
    const uint32_t nm = (uint32_t)mem.size();
    int rc;
    if (nm) {
        if ((rc = grow(ctx, ctx->bz_hmem, nm * sizeof(bz::Member), true))) return rc;
        if ((rc = grow(ctx, ctx->bz_mem, nm * sizeof(bz::Member), false))) return rc;
        if ((rc = grow(ctx, ctx->bz_match, in_total * 4 + 16, false))) return rc;
        if ((rc = grow(ctx, ctx->bz_work, slot_total, false))) return rc;
        if ((rc = grow(ctx, ctx->bz_out, slot_total, false))) return rc;
        if ((rc = grow(ctx, ctx->bz_size, (size_t)(nm + 1) * 4, false))) return rc;
        if ((rc = grow(ctx, ctx->bz_hsize, (size_t)(nm + 1) * 4, true))) return rc;
        memcpy(ctx->bz_hmem.p, mem.data(), nm * sizeof(bz::Member));
        CK(cudaMemcpyAsync(ctx->bz_mem.p, ctx->bz_hmem.p, nm * sizeof(bz::Member), cudaMemcpyHostToDevice, st));
        bz::DeflateArgs a;
        a.mem = (const bz::Member *)ctx->bz_mem.p;
        a.n = nm;
        a.match = (uint32_t *)ctx->bz_match.p;
        a.work = (uint8_t *)ctx->bz_work.p;
        a.size = (uint32_t *)ctx->bz_size.p;
        a.table = (const uint32_t *)((const uint8_t *)ctx->gz_tabs.p + 512);
        for (int j = 0; j < 8; j++) a.op[j] = ctx->bz_op[j];
        bool timed;                                      // tdg_timing_*: the three as one
        if ((rc = timed_start(ctx, timed))) return rc;
        bz::bgzf_deflate<<<nm, bz::THREADS, sizeof(bz::Shared), st>>>(a);
        tdg::tile_scan<<<1, 1024, 0, st>>>(a.size, nm);
        bz::bgzf_pack<<<nm, 256, 0, st>>>(a.mem, a.work, a.size, (uint8_t *)ctx->bz_out.p);
        if (timed) CK(cudaEventRecord(ctx->tev[ctx->tev_used++], st));
        ctx->launches += 3;
    }
    if (!cp.empty()) {                                   // after the members have read the old tails
        if ((rc = grow(ctx, ctx->bz_hcopy, cp.size() * sizeof(bz::Copy), true))) return rc;
        if ((rc = grow(ctx, ctx->bz_copy, cp.size() * sizeof(bz::Copy), false))) return rc;
        memcpy(ctx->bz_hcopy.p, cp.data(), cp.size() * sizeof(bz::Copy));
        CK(cudaMemcpyAsync(ctx->bz_copy.p, ctx->bz_hcopy.p, cp.size() * sizeof(bz::Copy), cudaMemcpyHostToDevice, st));
        bz::bgzf_copy<<<(unsigned)cp.size(), 256, 0, st>>>((const bz::Copy *)ctx->bz_copy.p);
        ctx->launches += 1;
    }
    CK(cudaGetLastError());
    ctx->bz_off.assign(nbar + 1, 0);
    if ((rc = grow(ctx, ctx->bz_hout, 16, true))) return rc;
    if (nm) {
        const uint32_t *hsize = (const uint32_t *)ctx->bz_hsize.p;
        CK(cudaMemcpyAsync(ctx->bz_hsize.p, ctx->bz_size.p, (size_t)(nm + 1) * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const uint32_t total = hsize[nm];
        if ((rc = grow(ctx, ctx->bz_hout, (size_t)total + 16, true))) return rc;
        if (total) CK(cudaMemcpyAsync(ctx->bz_hout.p, ctx->bz_out.p, total, cudaMemcpyDeviceToHost, st));
        for (uint32_t b = 0; b <= nbar; b++) ctx->bz_off[b] = hsize[first[b]];
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    *out = (const uint8_t *)ctx->bz_hout.p;
    *out_off = ctx->bz_off.data();
    return TDG_OK;
}

int tdg_split_bgzf(tdg_ctx *ctx, int on)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_split) return fail(ctx, TDG_ERR_STATE, "tdg_split_begin has not been called");
    CK(cudaSetDevice(ctx->device));
    ctx->bz_on = false;
    if (!on) return TDG_OK;
    if ((rc = gz_tables(ctx))) return rc;                // the CRC-32 table
    if ((rc = grow(ctx, ctx->bz_tail, (size_t)ctx->sp_nbar * tdg::bz::BLOCK, false))) return rc;
    if (!ctx->bz_attr) {
        CK(cudaFuncSetAttribute(tdg::bz::bgzf_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tdg::bz::Shared)));
        for (int j = 0; j < 8; j++) ctx->bz_op[j] = (uint32_t)crc32_combine_gen((z_off_t)(tdg::bz::SEG << j));
        ctx->bz_attr = true;
    }
    ctx->bz_tail_len.assign(ctx->sp_nbar, 0);
    ctx->bz_on = true;
    return TDG_OK;
}

int tdg_bgzf_append(tdg_ctx *ctx, const uint8_t *bytes, const uint64_t *off, const uint8_t **out, const uint64_t **out_off)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_split || !ctx->bz_on) return fail(ctx, TDG_ERR_STATE, "tdg_split_bgzf has not been called");
    if (!off || !out || !out_off) return fail(ctx, TDG_ERR_ARG, "null argument");
    const uint32_t nbar = ctx->sp_nbar;
    std::vector<uint64_t> rel(nbar + 1);
    for (uint32_t b = 0; b <= nbar; b++) {
        if (b && off[b] < off[b - 1]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
        rel[b] = off[b] - off[0];
    }
    const uint64_t n = rel[nbar];
    if (n && !bytes) return fail(ctx, TDG_ERR_ARG, "null argument");
    if (n > ((uint64_t)1 << 30)) return fail(ctx, TDG_ERR_ARG, "tdg_bgzf_append: at most 1 GiB per call");
    CK(cudaSetDevice(ctx->device));
    if ((rc = grow(ctx, ctx->bz_src, n + 16, false))) return rc;
    if (n) CK(cudaMemcpyAsync(ctx->bz_src.p, bytes + off[0], n, cudaMemcpyHostToDevice, ctx->stream));
    return bgzf_run(ctx, (const uint8_t *)ctx->bz_src.p, rel.data(), false, out, out_off);
}

int tdg_bgzf_finish(tdg_ctx *ctx, const uint8_t **out, const uint64_t **out_off)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_split || !ctx->bz_on) return fail(ctx, TDG_ERR_STATE, "tdg_split_bgzf has not been called");
    if (!out || !out_off) return fail(ctx, TDG_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    return bgzf_run(ctx, nullptr, nullptr, true, out, out_off);
}

int tdg_split_begin(tdg_ctx *ctx, const char *barcodes, const uint32_t *bar_off, uint32_t nbar, uint32_t cutlen)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    ctx->have_split = false;
    ctx->have_split_count = false;       // its rows are per barcode of this split
    if (!ctx->have_trim) return fail(ctx, TDG_ERR_STATE, "tdg_set_trim has not been called");
    if (!ctx->have_bar) return fail(ctx, TDG_ERR_STATE, "tdg_begin_file has not been called");
    if (!bar_off || (!barcodes && nbar && bar_off[nbar] != bar_off[0])) return fail(ctx, TDG_ERR_ARG, "null argument");
    if (nbar == 0 || nbar > 8192) return fail(ctx, TDG_ERR_ARG, "tdg_split_begin: between 1 and 8192 barcodes");
    if (nbar != ctx->trim_nbar || ctx->max_row >= nbar)
        return fail(ctx, TDG_ERR_ARG, "barcode table, trim tables and barcode list disagree on the number of barcodes");
    for (uint32_t i = 0; i < nbar; i++)
        if (bar_off[i + 1] < bar_off[i]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
    CK(cudaSetDevice(ctx->device));
    // one blob: bar_off [nbar+1], bar_len [nbar], strings
    const size_t o_len = (nbar + 1) * sizeof(uint32_t), o_str = o_len + nbar * sizeof(uint32_t);
    const size_t nstr = bar_off[nbar] - bar_off[0];
    std::vector<uint8_t> blob(o_str + nstr + 16);
    uint32_t *po = (uint32_t *)blob.data(), *pl = (uint32_t *)(blob.data() + o_len);
    for (uint32_t i = 0; i <= nbar; i++) po[i] = bar_off[i] - bar_off[0];
    for (uint32_t i = 0; i < nbar; i++) pl[i] = bar_off[i + 1] - bar_off[i];
    if (nstr) memcpy(blob.data() + o_str, barcodes + bar_off[0], nstr);
    rc = grow(ctx, ctx->sp_tabs, blob.size(), false);
    if (rc) return rc;
    CK(cudaMemcpy(ctx->sp_tabs.p, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    ctx->sp_nbar = nbar;
    ctx->sp_cutlen = cutlen;
    ctx->have_split = true;
    ctx->bz_on = false;
    return TDG_OK;
}

// tdg_split_block (host bytes) and tdg_split_device (device bytes, optionally sizes only): one block
// through split_front, then either the offsets and bytes of every barcode's file (bar_tile_sums ->
// bar_tile_scan -> bar_bases -> split_write) or, with sizes_only, their sizes alone (split_tally).
// totals (may be null) receive the block's reads, reads with barcode and cut site and reads clipped.
static int split_run(tdg_ctx *ctx, const char *what, const uint8_t *bytes, cudaMemcpyKind kind, size_t n, int final_block,
                     uint64_t max_records, bool sizes_only, uint64_t *n_records, uint64_t *consumed, int *needs_host,
                     const uint8_t **out, const uint64_t **out_off, const uint8_t **flags, uint64_t *totals)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_split || !ctx->have_trim || !ctx->have_bar) return fail(ctx, TDG_ERR_STATE, "tdg_split_begin has not been called");
    if (!n_records || !consumed || !needs_host || !out || !out_off || !flags || (!bytes && n)) return fail(ctx, TDG_ERR_ARG, "null argument");
    if (n > ((size_t)1 << 30)) return fail(ctx, TDG_ERR_ARG, std::string(what) + ": at most 1 GiB per block");
    *n_records = 0;
    *consumed = 0;
    *needs_host = 0;
    *out = nullptr;
    *out_off = nullptr;
    *flags = nullptr;
    if (totals)
        for (int k = 0; k < 3; k++) totals[k] = 0;
    if (n == 0 || max_records == 0) return TDG_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint32_t nbar = ctx->sp_nbar;
    tdg::SplitWork w;
    uint64_t nrec = 0;
    uint32_t last_end = 0;
    unsigned long long *bar_total = nullptr;
    if (sizes_only) {
        // tally [nbar] bytes per barcode, [3] flag counts, complex flag
        unsigned long long *tally = nullptr;
        rc = split_front(ctx, bytes, kind, n, final_block, max_records, w, nrec, last_end, [&](uint64_t) {
            int rc;
            if ((rc = grow(ctx, ctx->sp_base, (size_t)(nbar + 4) * sizeof(unsigned long long), false))) return rc;
            if ((rc = grow(ctx, ctx->sp_hbase, (size_t)(nbar + 4) * sizeof(unsigned long long), true))) return rc;
            tally = (unsigned long long *)ctx->sp_base.p;
            w.complex_flag = (uint32_t *)(tally + nbar + 3);
            CK(cudaMemsetAsync(tally, 0, (size_t)(nbar + 3) * sizeof(unsigned long long), st));
            return TDG_OK;
        });
        if (rc || nrec == 0) return rc;
        const uint32_t grid = (uint32_t)std::min<uint64_t>((nrec + tdg::SPLIT_REC_TILE - 1) / tdg::SPLIT_REC_TILE, 1024);
        tdg::split_tally<<<grid, tdg::SPLIT_REC_TILE, nbar * sizeof(uint32_t), st>>>(w, tally);
        ctx->launches += 1;
        unsigned long long *h = (unsigned long long *)ctx->sp_hbase.p;
        CK(cudaMemcpyAsync(h, tally, (size_t)(nbar + 4) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        *n_records = nrec;
        *consumed = last_end >= n ? n : (uint64_t)last_end + 1;
        if ((uint32_t)h[nbar + 3] != 0) {
            *needs_host = 1;
            return TDG_OK;
        }
        if (totals)
            for (int k = 0; k < 3; k++) totals[k] = h[nbar + k];
        unsigned long long run = 0;                  // the sizes become offsets, in place
        for (uint32_t b = 0; b < nbar; b++) {
            const unsigned long long c = h[b];
            h[b] = run;
            run += c;
        }
        h[nbar] = run;
        *out_off = (const uint64_t *)h;
        return TDG_OK;
    }
    rc = split_front(ctx, bytes, kind, n, final_block, max_records, w, nrec, last_end, [&](uint64_t records) {
        const uint32_t n_rtiles = (uint32_t)((records + tdg::SPLIT_REC_TILE - 1) / tdg::SPLIT_REC_TILE);
        int rc;
        if ((rc = grow(ctx, ctx->sp_sums, (size_t)n_rtiles * nbar * sizeof(uint32_t), false))) return rc;
        // bar_total [nbar], bar_base [nbar + 1], complex flag
        if ((rc = grow(ctx, ctx->sp_base, (size_t)(2 * nbar + 2) * sizeof(unsigned long long), false))) return rc;
        if ((rc = grow(ctx, ctx->sp_hbase, (size_t)(nbar + 2) * sizeof(unsigned long long), true))) return rc;
        if ((rc = grow(ctx, ctx->sp_hflags, (size_t)records + 16, true))) return rc;
        bar_total = (unsigned long long *)ctx->sp_base.p;
        w.bar_base = bar_total + nbar;
        w.complex_flag = (uint32_t *)(bar_total + 2 * nbar + 1);
        w.n_rtiles = n_rtiles;
        w.tile_sums = (uint32_t *)ctx->sp_sums.p;
        return TDG_OK;
    });
    if (rc || nrec == 0) return rc;
    const uint32_t n_rtiles = w.n_rtiles;
    tdg::bar_tile_sums<<<n_rtiles, tdg::SPLIT_REC_TILE, nbar * sizeof(uint32_t), st>>>(w);
    tdg::bar_tile_scan<<<(nbar + 255) / 256, 256, 0, st>>>(w, bar_total);
    tdg::bar_bases<<<1, 32, 0, st>>>(bar_total, w.bar_base, nbar);
    ctx->launches += 3;
    unsigned long long *hbase = (unsigned long long *)ctx->sp_hbase.p;
    CK(cudaMemcpyAsync(hbase, w.bar_base, (size_t)(nbar + 2) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    *n_records = nrec;
    *consumed = last_end >= n ? n : (uint64_t)last_end + 1;
    if ((uint32_t)hbase[nbar + 1] != 0) {            // the complex flag sits right behind bar_base[nbar]
        *needs_host = 1;
        return TDG_OK;
    }

    // ---- the bytes of every barcode's file
    const size_t total_out = (size_t)hbase[nbar];
    if ((rc = grow(ctx, ctx->sp_out, total_out + 16, false))) return rc;
    w.out = (uint8_t *)ctx->sp_out.p;
    tdg::split_write<<<n_rtiles, tdg::SPLIT_REC_TILE, nbar * sizeof(uint32_t), st>>>(w);
    ctx->launches += 1;
    if (ctx->bz_on) {                                // the bytes stay on the device and become members
        CK(cudaMemcpyAsync(ctx->sp_hflags.p, w.flags, nrec, cudaMemcpyDeviceToHost, st));
        if ((rc = bgzf_run(ctx, w.out, (const uint64_t *)hbase, false, out, out_off))) return rc;
        *flags = (const uint8_t *)ctx->sp_hflags.p;
        return TDG_OK;
    }
    if ((rc = grow(ctx, ctx->sp_hout, total_out + 16, true))) return rc;
    if (total_out) CK(cudaMemcpyAsync(ctx->sp_hout.p, w.out, total_out, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ctx->sp_hflags.p, w.flags, nrec, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    *out = (const uint8_t *)ctx->sp_hout.p;
    *out_off = (const uint64_t *)hbase;
    *flags = (const uint8_t *)ctx->sp_hflags.p;
    if (totals) {
        totals[0] = nrec;
        for (uint64_t r = 0; r < nrec; r++) {
            totals[1] += (*flags)[r] & tdg::SPLIT_FLAG_BAR ? 1 : 0;
            totals[2] += (*flags)[r] & tdg::SPLIT_FLAG_CLIP ? 1 : 0;
        }
    }
    return TDG_OK;
}

int tdg_split_block(tdg_ctx *ctx, const uint8_t *bytes, size_t n, int final_block, uint64_t max_records,
                    uint64_t *n_records, uint64_t *consumed, int *needs_host, const uint8_t **out,
                    const uint64_t **out_off, const uint8_t **flags)
{
    return split_run(ctx, "tdg_split_block", bytes, cudaMemcpyHostToDevice, n, final_block, max_records, false, n_records,
                     consumed, needs_host, out, out_off, flags, nullptr);
}

int tdg_split_device(tdg_ctx *ctx, const void *dev_bytes, size_t n, int final_block, uint64_t max_records, int sizes_only,
                     uint64_t *n_records, uint64_t *consumed, int *needs_host, const uint8_t **out,
                     const uint64_t **out_off, const uint8_t **flags, uint64_t totals[3])
{
    if (ctx && ctx->bz_on) return fail(ctx, TDG_ERR_STATE, "tdg_split_device: BGZF output is on (tdg_split_bgzf)");
    if (ctx && !totals) return fail(ctx, TDG_ERR_ARG, "null argument");
    return split_run(ctx, "tdg_split_device", (const uint8_t *)dev_bytes, cudaMemcpyDeviceToDevice, n, final_block,
                     max_records, sizes_only != 0, n_records, consumed, needs_host, out, out_off, flags, totals);
}

int tdg_split_count_begin(tdg_ctx *ctx, const char *bases, const uint32_t *off, const uint32_t *tag_off, uint32_t npat,
                          uint32_t flags, const int32_t *row_of_barcode)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    ctx->have_split_count = false;
    if (!ctx->have_tags) return fail(ctx, TDG_ERR_STATE, "tdg_set_tags has not been called");
    if (!ctx->d_matrix) return fail(ctx, TDG_ERR_STATE, "tdg_set_matrix / tdg_bind_matrix has not been called");
    if (!ctx->have_split) return fail(ctx, TDG_ERR_STATE, "tdg_split_begin has not been called");
    if (!off || !tag_off || !row_of_barcode) return fail(ctx, TDG_ERR_ARG, "null argument");
    const uint32_t nbar = ctx->sp_nbar;
    uint32_t max_row = 0;
    for (uint32_t b = 0; b < nbar; b++) {
        if (row_of_barcode[b] < 0 || (uint32_t)row_of_barcode[b] >= ctx->rows)
            return fail(ctx, TDG_ERR_ARG, "tdg_split_count_begin: a barcode row lies outside the matrix");
        max_row = std::max(max_row, (uint32_t)row_of_barcode[b]);
    }
    // the table's own rows are never read: a hit goes to the row of the record's stage-1 barcode
    const std::vector<int32_t> zero(npat, 0);
    std::vector<uint8_t> blob;
    std::string why = tdg::build_bar_table(bases, off, zero.data(), tag_off, npat, flags, blob);
    if (!why.empty()) return fail(ctx, TDG_ERR_ARG, "tdg_split_count_begin: " + why);
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));          // earlier kernels read the old tables
    if ((rc = grow(ctx, ctx->sc_bar, round_up(blob.size(), 16), false)) || (rc = grow(ctx, ctx->sc_rows, nbar * sizeof(int32_t), false)) ||
        (rc = grow_exact(ctx, ctx->sc_tot, 5 * sizeof(unsigned long long), false)) ||
        (rc = grow_exact(ctx, ctx->sc_htot, 5 * sizeof(unsigned long long), true)))
        return rc;
    CK(cudaMemcpy(ctx->sc_bar.p, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->sc_rows.p, row_of_barcode, nbar * sizeof(int32_t), cudaMemcpyHostToDevice));
    ctx->sc_max_row = max_row;
    ctx->have_split_count = true;
    return TDG_OK;
}

// tdg_split_count_block (host bytes) and tdg_split_count_device (device bytes): one block through
// split_front and split_count.
static int split_count_run(tdg_ctx *ctx, const char *what, const uint8_t *bytes, cudaMemcpyKind kind, size_t n,
                           int final_block, uint64_t max_records, uint64_t *n_records, uint64_t *consumed, int *needs_host,
                           uint64_t totals[4])
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if ((rc = split_count_ready(ctx))) return rc;
    if (!n_records || !consumed || !needs_host || !totals || (!bytes && n)) return fail(ctx, TDG_ERR_ARG, "null argument");
    if (n > ((size_t)1 << 30)) return fail(ctx, TDG_ERR_ARG, std::string(what) + ": at most 1 GiB per block");
    *n_records = 0;
    *consumed = 0;
    *needs_host = 0;
    for (int k = 0; k < 4; k++) totals[k] = 0;
    if (n == 0 || max_records == 0) return TDG_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    unsigned long long *d_tot = (unsigned long long *)ctx->sc_tot.p;     // totals [4], complex flag
    tdg::SplitWork w;
    uint64_t nrec = 0;
    uint32_t last_end = 0;
    bool timed;                                      // tdg_timing_*: the block's upload and kernels as one
    if ((rc = timed_start(ctx, timed))) return rc;
    rc = split_front(ctx, bytes, kind, n, final_block, max_records, w, nrec, last_end, [&](uint64_t) {
        w.complex_flag = (uint32_t *)(d_tot + 4);
        CK(cudaMemsetAsync(d_tot, 0, 4 * sizeof(unsigned long long), st));
        return TDG_OK;
    });
    if (!rc && nrec) {
        tdg::split_count<<<(unsigned)((nrec + 255) / 256), 256, 0, st>>>(w, split_count_args(ctx), d_tot);
        ctx->launches += 1;
    }
    if (timed) CK(cudaEventRecord(ctx->tev[ctx->tev_used++], st));
    if (rc || nrec == 0) return rc;
    const unsigned long long *h = (const unsigned long long *)ctx->sc_htot.p;
    CK(cudaMemcpyAsync(ctx->sc_htot.p, d_tot, 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    *n_records = nrec;
    *consumed = last_end >= n ? n : (uint64_t)last_end + 1;
    if ((uint32_t)h[4] != 0) {                       // split_count left the matrix alone
        *needs_host = 1;
        return TDG_OK;
    }
    for (int k = 0; k < 4; k++) totals[k] = h[k];
    return TDG_OK;
}

int tdg_split_count_block(tdg_ctx *ctx, const uint8_t *bytes, size_t n, int final_block, uint64_t max_records,
                          uint64_t *n_records, uint64_t *consumed, int *needs_host, uint64_t totals[4])
{
    return split_count_run(ctx, "tdg_split_count_block", bytes, cudaMemcpyHostToDevice, n, final_block, max_records, n_records,
                           consumed, needs_host, totals);
}

int tdg_split_count_device(tdg_ctx *ctx, const void *dev_bytes, size_t n, int final_block, uint64_t max_records,
                           uint64_t *n_records, uint64_t *consumed, int *needs_host, uint64_t totals[4])
{
    return split_count_run(ctx, "tdg_split_count_device", (const uint8_t *)dev_bytes, cudaMemcpyDeviceToDevice, n, final_block,
                           max_records, n_records, consumed, needs_host, totals);
}

int tdg_split_count_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, const int32_t *bar, uint32_t n, int32_t *col_out)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if ((rc = split_count_ready(ctx))) return rc;
    if (n == 0) return TDG_OK;
    if (!off || !bar || !col_out || (!seqs && off[n] != off[0])) return fail(ctx, TDG_ERR_ARG, "null argument");
    for (uint32_t i = 0; i < n; i++) {
        if (bar[i] < 0 || (uint32_t)bar[i] >= ctx->sp_nbar) return fail(ctx, TDG_ERR_ARG, "barcode index out of range");
        if (off[i + 1] < off[i]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
    }
    CK(cudaSetDevice(ctx->device));
    return batch_run(ctx, "tdg_split_count_batch", seqs, off, n, {{bar, nullptr, n * sizeof(int32_t)}, {nullptr, col_out, n * sizeof(int32_t)}},
                     [&](const uint8_t *d, const unsigned long long *d_off, uint8_t *const *part) {
                         tdg::split_count_batch<<<(n + 127) / 128, 128, 0, ctx->stream>>>(d, d_off, (const int32_t *)part[0], n,
                                                                                         split_count_args(ctx), (int32_t *)part[1]);
                     });
}

// ---------------------------------------------------------------------------
// The host feed on its own (tdg_feed.h): uncompressed bytes of a plain / gzip / BGZF file.

struct tdg_feed {
    tdg::Feeder f;
};

int tdg_feed_open(tdg_feed **out, const char *path, int gz)
{
    if (!out || !path) return fail(nullptr, TDG_ERR_ARG, "null argument");
    *out = nullptr;
    tdg_feed *h = new (std::nothrow) tdg_feed();
    if (!h) return fail(nullptr, TDG_ERR_NOMEM, "out of memory");
    int rc = h->f.open(path, gz != 0);
    if (rc) {
        fail(nullptr, rc, h->f.error());
        delete h;
        return rc;
    }
    *out = h;
    return TDG_OK;
}

long long tdg_feed_read(tdg_feed *h, void *dst, size_t cap)
{
    if (!h || (!dst && cap)) return fail(nullptr, TDG_ERR_ARG, "null argument");
    if (cap == 0) return 0;
    long long r = h->f.fill((uint8_t *)dst, cap);
    if (r < 0) fail(nullptr, (int)r, h->f.error());
    return r;
}

void tdg_feed_close(tdg_feed *h) { delete h; }

int tdg_match_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, uint32_t n, int32_t *row_out, int32_t *col_out)
{
    int rc = need_device(ctx);
    if (rc) return rc;
    if (!ctx->have_tags) return fail(ctx, TDG_ERR_STATE, "tdg_set_tags has not been called");
    if (!ctx->have_bar) return fail(ctx, TDG_ERR_STATE, "tdg_begin_file has not been called");
    if (n == 0) return TDG_OK;
    if (!off || !row_out || !col_out || (!seqs && off[n] != off[0])) return fail(ctx, TDG_ERR_ARG, "null argument");
    for (uint32_t i = 0; i < n; i++)
        if (off[i + 1] < off[i]) return fail(ctx, TDG_ERR_ARG, "offsets must be non-decreasing");
    CK(cudaSetDevice(ctx->device));
    return batch_run(ctx, "tdg_match_batch", seqs, off, n, {{nullptr, row_out, n * sizeof(int32_t)}, {nullptr, col_out, n * sizeof(int32_t)}},
                     [&](const uint8_t *d, const unsigned long long *d_off, uint8_t *const *part) {
                         tdg::MatchArgs a;
                         a.seqs = d;
                         a.off = d_off;
                         a.n = n;
                         a.bar = (const tdg::BarTable *)ctx->d_bar.p;
                         a.tags = ctx->tags.t;
                         a.tags.entries = (const tdg::TagEntry *)ctx->d_entries.p;
                         a.tags.ext = (const uint64_t *)ctx->d_ext.p;
                         a.row_out = (int32_t *)part[0];
                         a.col_out = (int32_t *)part[1];
                         tdg::match_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(a);
                     });
}

// ---------------------------------------------------------------------------
// CSV output (host threads), csrc/tdg_csv.h.  No context needed: errors go to the
// message returned by tdg_last_error(NULL).

int tdg_write_counts_csv(const char *path, const int32_t *matrix, uint32_t rows, uint32_t cols, const char *header,
                         size_t header_len, const char *labels, const uint64_t *label_off, int threads)
{
    if (!path || (!matrix && rows && cols) || !header || !label_off || (!labels && rows && label_off[rows] != label_off[0]))
        return fail(nullptr, TDG_ERR_ARG, "null argument");
    std::string why = tdg::write_table(path, header, header_len, rows, cols, labels, label_off, threads,
                                       [=](char *p, uint32_t r, uint32_t c) { return tdg::put_int(p, matrix[(size_t)r * cols + c]); });
    if (!why.empty()) return fail(nullptr, TDG_ERR_IO, why);
    return TDG_OK;
}

int tdg_write_geno_csv(const char *path, const int32_t *matrix, uint32_t rows, uint32_t cols, const uint32_t *col0,
                       const uint32_t *col1, uint32_t nmarkers, const char *header, size_t header_len, const char *labels,
                       const uint64_t *label_off, int threads)
{
    if (!path || (!matrix && rows && cols) || !header || !label_off || (nmarkers && (!col0 || !col1)))
        return fail(nullptr, TDG_ERR_ARG, "null argument");
    for (uint32_t m = 0; m < nmarkers; m++)
        if (col0[m] >= cols || col1[m] >= cols) return fail(nullptr, TDG_ERR_ARG, "marker column outside the matrix");
    std::string why = tdg::write_table(path, header, header_len, rows, nmarkers, labels, label_off, threads,
                                       [=](char *p, uint32_t r, uint32_t m) {
                                           // writeDiploidGeno, tagdigger_fun.py:1160-1167
                                           const bool a = matrix[(size_t)r * cols + col0[m]] > 0, b = matrix[(size_t)r * cols + col1[m]] > 0;
                                           if (a || b) *p++ = a && b ? '1' : (a ? '0' : '2');
                                           return p;
                                       });
    if (!why.empty()) return fail(nullptr, TDG_ERR_IO, why);
    return TDG_OK;
}

}  // extern "C"
