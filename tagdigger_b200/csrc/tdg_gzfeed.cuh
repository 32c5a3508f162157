// Host side of the device gzip feed: rounds, uploads, the checks against trailers, the hand-over to
// the host feeder, the read limit, and the two sinks (counting; copying out).  The kernels are in
// tdg_gzdev.cuh, the per-lane inflater in tdg_gzlane.h, the chain of a round in tdg_gzchain.h.
//
// This file is PART OF tdg_api.cu (included there, inside its anonymous namespace, behind the
// definitions of tdg_ctx, Buf, fail, CK, grow, make_event, launch_chunk, line_cut, ensure_slots): it is a
// separate file for the reader's sake, not a separate unit.
// ---------------------------------------------------------------------------
// Device-side gzip feed (tdg_gzlane.h, tdg_gzchain.h, tdg_gzdev.cuh)

constexpr int TDG_STOP_ROUND = -1000;       // (internal) the sink does not want this round

struct GzStats {
    uint32_t rounds = 0, chunks = 0, accepted = 0;
    double ms_upload = 0, ms_scan = 0, ms_decode = 0, ms_host = 0, ms_resolve = 0, ms_sink = 0;
};

// The read limit of find_tags_fastq (maxreads, default 5e9: tagdigger_fun.py:192, :272-273) on the
// host side of tdg_count_file.  The kernels apply the limit exactly whatever the host does; what the
// host owes the reference is to STOP READING at the limit (a defect behind it is never met).  Looking
// for the limit's line end costs a pass over every byte, so it is done only where the limit can be:
// a piece of n bytes holds at most n line ends, and while (line ends so far, at most) + n stays below
// the limit's line the piece goes through untouched.  When that bound is used up, the exact number of
// lines is read back from the device (a few times per 20 GB at the default limit) -- and only when
// the limit really lies within reach are pieces scanned (tdg::LineLimit).
struct LimitState {
    bool has = false;
    uint64_t line = 0;           // the limit's line end: number 4 * maxreads - 2
    uint64_t lines_ub = 0;       // line ends handed to the device so far, at most
    bool careful = false;        // pieces are scanned
    tdg::LineLimit ll;
    uint8_t last_byte = 0;       // of the text so far (a '\r' there may still end a line)

    void init(uint64_t reads_limit, size_t chunk_bytes)
    {
        has = reads_limit < ((uint64_t)1 << 60);
        line = has ? (reads_limit ? 4 * reads_limit - 2 : 1) : 0;
        if (has && line <= chunk_bytes) {                    // within reach of the first piece: scan from the start
            careful = true;
            ll.remaining = line;
        }
    }
};

// May `nbytes` more bytes of text go to the device without a look?  1 yes, 0 no (lim.careful is set and
// lim.ll counts down to the limit's line from here), negative: error.
int limit_admits(tdg_ctx *ctx, LimitState &lim, size_t nbytes)
{
    if (!lim.has) return 1;
    if (lim.careful) return 0;
    if (lim.lines_ub + nbytes < lim.line) {
        lim.lines_ub += nbytes;
        return 1;
    }
    uint64_t t[4];
    int rc = tdg_file_totals(ctx, t);                        // (synchronises) t[3]: line ends counted so far, exactly
    if (rc) return rc;
    lim.lines_ub = t[3];
    if (lim.lines_ub + nbytes < lim.line) {
        lim.lines_ub += nbytes;
        return 1;
    }
    lim.careful = true;
    lim.ll.remaining = lim.line - t[3];
    lim.ll.prev_cr = lim.last_byte == '\r';
    return 0;
}

// what happens to a round's text: counted (tdg_count_file) or copied out (tdg_gz_inflate_host)
struct GzSink {
    virtual ~GzSink() {}
    // d_buf[0 .. carry) = bytes kept from the round before, d_buf[carry .. carry + len) = new text.
    // Sets `carry` to the number of bytes it wants to see again, in front of the next round's text
    // (they must be at d_buf[0 ..) when it returns -- stream order).
    virtual int text(tdg_ctx *ctx, uint8_t *d_buf, size_t &carry, size_t len) = 0;
    // Asked before a round's text is accepted: 1 go on, 0 the device feed must stop in front of this
    // round (a read limit within reach: the host feeder takes over and stops at the limit), < 0 error.
    virtual int may_take(tdg_ctx *, size_t) { return 1; }
};

int gz_io_threads()
{
    int t = 16;
    if (const char *e = getenv("TDG_IO_THREADS")) t = std::max(1, atoi(e));
    unsigned hw = std::thread::hardware_concurrency();
    if (hw && t > (int)hw) t = (int)hw;
    return t;
}

bool gz_pread_parallel(int fd, uint8_t *dst, size_t n, uint64_t off, int threads)
{
    int nt = (int)std::min<size_t>((size_t)threads, std::max<size_t>(1, n >> 22));
    std::vector<char> ok(nt, 1);
    auto work = [&](int t) {
        size_t lo = n / nt * t, hi = t == nt - 1 ? n : n / nt * (t + 1);
        while (lo < hi) {
            ssize_t r = pread(fd, dst + lo, hi - lo, (off_t)(off + lo));
            if (r <= 0) { ok[t] = 0; return; }
            lo += (size_t)r;
        }
    };
    tdg::Pool::get().run(nt, work);
    for (char c : ok)
        if (!c) return false;
    return true;
}

int gz_tables(tdg_ctx *ctx)
{
    if (ctx->gz_tables) return TDG_OK;
    // [kraft3 512][crc table 256 x u32][window 32768]
    int rc = grow(ctx, ctx->gz_tabs, 512 + 1024 + tdg::gzl::WIN, false);
    if (rc) return rc;
    std::vector<uint8_t> blob(512 + 1024);
    tdg::gzl::make_kraft3(blob.data());
    uint32_t *tab = (uint32_t *)(blob.data() + 512);
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? 0xEDB88320u : 0u);
        tab[i] = c;
    }
    CK(cudaMemcpy(ctx->gz_tabs.p, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    for (int j = 0; j < 8; j++) ctx->gz_op[j] = (uint32_t)crc32_combine_gen((z_off_t)(tdg::gzd::SUB << j));
    for (Event &ev : ctx->gz_up)
        if ((rc = make_event(ctx, ev))) return rc;
    if ((rc = make_event(ctx, ctx->gz_pre))) return rc;
    CK(cudaFuncSetAttribute(tdg::gzd::gz_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tdg::gzd::DEC_SMEM));
    CK(cudaFuncSetAttribute(tdg::gzd::gz_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tdg::gzd::SCAN_SMEM));
    ctx->gz_tables = true;
    return TDG_OK;
}

// A mapped file (the device feeds parse headers and trailers in it; the bytes themselves go through pread)
struct GzMap {
    int fd = -1;
    const uint8_t *p = nullptr;
    size_t n = 0;
    ~GzMap()
    {
        if (p) munmap(const_cast<uint8_t *>(p), n);
        if (fd >= 0) ::close(fd);
    }
};

// file bytes [off, end) -> compressed buffer `which` (zero padded), through the three pinned buffers, on `stream`
int gz_upload(tdg_ctx *ctx, const GzMap &map, const char *path, int threads, int &up_i, int which, size_t off, size_t end,
              cudaStream_t stream)
{
    Buf &g = which ? ctx->gz_comp2 : ctx->gz_comp;
    const size_t nb = end - off, padded = (nb + 3) / 4 * 4 + 256;
    int rc = grow(ctx, g, padded, false);
    if (rc) return rc;
    const size_t piece = ctx->chunk_bytes;                  // the size of the pinned file buffers
    for (size_t at = 0; at < nb; at += piece, up_i = (up_i + 1) % 3) {
        const size_t m = std::min(piece, nb - at);
        uint8_t *pinned = (uint8_t *)ctx->file_buf[0][up_i].p;
        CK(cudaEventSynchronize(ctx->gz_up[up_i]));
        if (!gz_pread_parallel(map.fd, pinned, m, off + at, threads))
            return fail(ctx, TDG_ERR_IO, std::string("read error on ") + path);
        CK(cudaMemcpyAsync((uint8_t *)g.p + at, pinned, m, cudaMemcpyHostToDevice, stream));
        CK(cudaEventRecord(ctx->gz_up[up_i], stream));
    }
    CK(cudaMemsetAsync((uint8_t *)g.p + nb, 0, padded - nb, stream));
    return TDG_OK;
}

using GzClock = std::chrono::steady_clock;
double gz_ms(GzClock::time_point a, GzClock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); }

// One device feed of one file: what its rounds share.  A round ends with its text at the sink.  Before
// that, TDG_ERR_NOMEM (a buffer that cannot be had) and TDG_STOP_ROUND (the sink does not want the text)
// are not the file's fault: the host feeder continues at the state the round began in (gz_device_feed).
struct GzFeed {
    tdg_ctx *ctx;
    const char *path;
    GzSink &sink;
    size_t &carry;
    GzStats &stats;
    tdg::Utf8State *u8;
    GzMap map;
    uint32_t max_chunks = 0;
    size_t fixed_chunk = 0;
    uint32_t fixed_cap = 0;
    bool debug = false;
    int threads = 0;
    int up_i = 0;                // the pinned buffer gz_upload fills next
    bool sunk = false;           // the sink has had the round's text: a failure from here on is the call's
    bool done = false;           // the device fed the whole file
    bool handover = false;       // the host feeder continues at the position below
    // a stream: where it stands, and the next round's bytes when they were read ahead
    tdg::gzc::Stream st;
    int cur = 0;                 // which compressed buffer the round reads
    bool pre_valid = false;      // the other one holds [pre_off, pre_end) of the file
    size_t pre_off = 0, pre_end = 0;
    // BGZF: the next member, and the bytes of text in front of it
    size_t off = 0;
    uint64_t delivered = 0;

    int upload(int which, size_t from, size_t end, cudaStream_t stream) { return gz_upload(ctx, map, path, threads, up_i, which, from, end, stream); }
    int to_sink(uint64_t text_len)
    {
        sunk = true;
        return sink.text(ctx, (uint8_t *)ctx->gz_text.p, carry, (size_t)text_len);
    }
};

// what gz_scan and gz_decode read of a round (nb compressed bytes at `in`) and where the lanes put their tokens and reports
tdg::gzd::RoundArgs gz_round_args(tdg_ctx *ctx, const void *in, size_t nb, uint32_t nchunks, uint32_t symcap, uint32_t tokcap)
{
    using namespace tdg;
    gzd::RoundArgs a;
    memset(&a, 0, sizeof(a));
    a.in = (const uint32_t *)in;
    a.nwords = (nb + 3) / 4;
    a.in_bits = (uint64_t)nb * 8;
    a.nchunks = nchunks;
    a.symcap = symcap;
    a.tokcap = tokcap;
    a.syms = (uint16_t *)ctx->gz_syms.p;
    a.meta = (gzl::Meta *)ctx->gz_meta.p;
    a.cold = (uint16_t *)ctx->gz_cold.p;
    return a;
}

// ---- the text stage: the steps both formats run alike, from the tokens of a round's chunks (or members) to the sink

// gz_text[carry ..) must take text_len more bytes (and the counting kernel's tiles and halo); the carried bytes stay in front
int gz_text_room(tdg_ctx *ctx, size_t carry, uint64_t text_len)
{
    const size_t need = round_up(carry + text_len, TDG_TILE_BYTES) + TDG_HALO_BYTES + 64;
    if (need <= ctx->gz_text.cap) return TDG_OK;
    int rc;
    if (carry) {
        if ((rc = grow(ctx, ctx->gz_carry, carry, false))) return rc;
        CK(cudaMemcpyAsync(ctx->gz_carry.p, ctx->gz_text.p, carry, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    if ((rc = grow(ctx, ctx->gz_text, need, false))) return rc;
    if (carry) CK(cudaMemcpyAsync(ctx->gz_text.p, ctx->gz_carry.p, carry, cudaMemcpyDeviceToDevice, ctx->stream));
    return TDG_OK;
}

// tokens -> symbols: the ntok[k] tokens of chunk k in gz_syms (tokcap apart) become its symbols in gz_sym2 (symcap apart)
int gz_expand_tokens(tdg_ctx *ctx, const std::vector<uint32_t> &ntok, uint32_t tokcap, uint32_t symcap)
{
    using namespace tdg;
    CK(cudaMemcpyAsync(ctx->gz_ntok.p, ntok.data(), ntok.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));      // (ntok is the caller's)
    gzd::ExpandArgs ea;
    ea.tok = (uint16_t *)ctx->gz_syms.p;
    ea.syms = (uint16_t *)ctx->gz_sym2.p;
    ea.tokcap = tokcap;
    ea.symcap = symcap;
    ea.ntok = (const uint32_t *)ctx->gz_ntok.p;
    ea.accepted = (uint32_t)ntok.size();
    gzd::gz_expand<<<(ea.accepted + gzd::EXP_WARPS - 1) / gzd::EXP_WARPS, gzd::EXP_WARPS * 32, 0, ctx->stream>>>(ea);
    CK(cudaGetLastError());
    ctx->launches++;
    return TDG_OK;
}

// symbols -> the round's text at gz_text + carry.  gz_crc gets the raw CRC-32 of each of its `pieces` pieces and,
// behind them, a flag with the high bit of every byte.
int gz_resolve_text(tdg_ctx *ctx, uint32_t symcap, const uint64_t *text_off, uint32_t accepted, size_t carry, uint64_t text_len,
                    uint32_t pieces)
{
    using namespace tdg;
    uint32_t *d_flag = (uint32_t *)ctx->gz_crc.p + pieces;
    CK(cudaMemsetAsync(d_flag, 0, 4, ctx->stream));
    gzd::ResArgs ra;
    ra.syms = (const uint16_t *)ctx->gz_sym2.p;
    ra.symcap = symcap;
    ra.text_off = text_off;
    ra.accepted = accepted;
    ra.ptrs = (const uint32_t *)ctx->gz_windows.p;
    ra.text = (uint8_t *)ctx->gz_text.p + carry;
    ra.text_len = text_len;
    ra.crc = (uint32_t *)ctx->gz_crc.p;
    ra.flag = d_flag;
    ra.table = (const uint32_t *)((uint8_t *)ctx->gz_tabs.p + 512);
    for (int j = 0; j < 8; j++) ra.op[j] = ctx->gz_op[j];
    gzd::gz_resolve<<<pieces, gzd::RES_THREADS, 0, ctx->stream>>>(ra);
    CK(cudaGetLastError());
    ctx->launches++;
    return TDG_OK;
}

// text mode: bytes >= 0x80 (high_flag: the resolve kernel saw one) must form valid UTF-8 (open(f, 'rt'))
int gz_check_utf8(GzFeed &f, uint32_t high_flag, uint64_t text_len)
{
    tdg_ctx *ctx = f.ctx;
    if (!f.u8) return TDG_OK;
    if ((high_flag & 0x80u) || f.u8->need) {
        std::vector<uint8_t> host(text_len);
        CK(cudaMemcpy(host.data(), (uint8_t *)ctx->gz_text.p + f.carry, text_len, cudaMemcpyDeviceToHost));
        long long bad = tdg::utf8_feed(*f.u8, host.data(), host.size());
        if (bad >= 0) return fail(ctx, TDG_ERR_UTF8, "position " + std::to_string(bad) + ": invalid UTF-8 in " + f.path);
    } else {
        f.u8->offset += text_len;
    }
    return TDG_OK;
}

// A round of BGZF (bgzip): gzip members of at most 64 KiB of text that carry their compressed size in a 'BC'
// extra field -- every member is its own deflate stream, so nothing is speculative here: the host
// walks the member headers, one lane inflates one member from its first bit to its final block
// (gz_decode in member mode), gz_expand and gz_resolve lay the text out, gz_member_crc takes every
// member's CRC-32, and the host holds length, end position and CRC against the member's trailer.
// A member that fails any of that is what the host feeder calls a corrupt BGZF member; a member
// header that is not BGZF (or a truncated one) ends the device feed, the host feeder continues there.
int gz_bgzf_round(GzFeed &f)
{
    using namespace tdg;
    struct Member {
        size_t off;
        uint32_t hlen, csize, isize, crc;
    };
    tdg_ctx *ctx = f.ctx;
    const GzMap &map = f.map;
    const uint32_t symcap = 65536 + 512, tokcap = 65536 + 64;
    int rc;
    // ---- the members of this round
    auto t0 = GzClock::now();
    std::vector<Member> mem;
    size_t end = f.off;
    while (end < map.n && mem.size() < f.max_chunks && end - f.off < ((size_t)1 << 30)) {
        uint32_t csize = 0, hlen = 0;
        if (!Feeder::bgzf_member(map.p + end, std::min<size_t>(map.n - end, 1024), csize, hlen) || end + csize > map.n) {
            f.handover = true;
            break;
        }
        Member m;
        m.off = end;
        m.hlen = hlen;
        m.csize = csize;
        memcpy(&m.crc, map.p + end + csize - 8, 4);
        memcpy(&m.isize, map.p + end + csize - 4, 4);
        if (m.isize > 65536) {
            f.handover = true;
            break;
        }
        mem.push_back(m);
        end += csize;
    }
    if (mem.empty()) return TDG_OK;
    const uint32_t n = (uint32_t)mem.size();
    const size_t nb = end - f.off;
    if ((rc = f.upload(0, f.off, end, ctx->stream))) return rc;
    if ((rc = grow(ctx, ctx->gz_syms, (size_t)n * tokcap * 2, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_sym2, (size_t)n * symcap * 2, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_meta, (size_t)n * sizeof(gzl::Meta), false))) return rc;
    if ((rc = grow(ctx, ctx->gz_hmeta, (size_t)n * sizeof(gzl::Meta), true))) return rc;
    if ((rc = grow(ctx, ctx->gz_cold, (size_t)(n + 8) * gzl::COLD_U16 * 2, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_offs, ((size_t)n * 3 + 1) * 8, false))) return rc;       // [n] start bits, [n] end bits, [n + 1] text offsets
    if ((rc = grow(ctx, ctx->gz_lens, (size_t)n * 4, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_ntok, (size_t)n * 4, false))) return rc;
    std::vector<uint64_t> bits(2 * (size_t)n), text_off(n + 1, 0);
    std::vector<uint32_t> lens(n);
    for (uint32_t k = 0; k < n; k++) {
        bits[k] = (uint64_t)(mem[k].off + mem[k].hlen - f.off) * 8;
        bits[n + k] = (uint64_t)(mem[k].off + mem[k].csize - 8 - f.off) * 8;
        lens[k] = mem[k].isize;
        text_off[k + 1] = text_off[k] + mem[k].isize;
    }
    const uint64_t text_len = text_off[n];
    uint64_t *d_bits = (uint64_t *)ctx->gz_offs.p;
    uint64_t *d_toff = d_bits + 2 * (size_t)n;
    CK(cudaMemcpyAsync(d_bits, bits.data(), bits.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_toff, text_off.data(), text_off.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->gz_lens.p, lens.data(), lens.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    gzd::RoundArgs a = gz_round_args(ctx, ctx->gz_comp.p, nb, n, symcap, tokcap);
    a.m_start = d_bits;
    a.m_end = d_bits + n;
    gzd::gz_decode<<<(n + gzd::DEC_THREADS - 1) / gzd::DEC_THREADS, gzd::DEC_THREADS, gzd::DEC_SMEM, ctx->stream>>>(a);
    CK(cudaGetLastError());
    gzl::Meta *meta = (gzl::Meta *)ctx->gz_hmeta.p;
    CK(cudaMemcpyAsync(meta, ctx->gz_meta.p, (size_t)n * sizeof(gzl::Meta), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    auto t1 = GzClock::now();
    // ---- every member must have ended with its final block, right in front of its trailer, at its length
    std::vector<uint32_t> ntok(n);
    for (uint32_t k = 0; k < n; k++) {
        const gzl::Meta &c = meta[k];
        const bool good = c.flags == (gzl::F_FOUND | gzl::F_FINAL) && c.out_len == mem[k].isize && (c.end_bit + 7) / 8 * 8 == bits[n + k];
        if (!good) return fail(ctx, TDG_ERR_GZIP, std::string("gzip error in ") + f.path + ": corrupt BGZF member");
        ntok[k] = c.ntok;
    }
    if (text_len) {
        const int go = f.sink.may_take(ctx, (size_t)text_len);
        if (go < 0) return go;
        if (go == 0) return TDG_STOP_ROUND;
        const uint32_t pieces = (uint32_t)((text_len + gzd::PIECE - 1) / gzd::PIECE);
        if ((rc = grow(ctx, ctx->gz_crc, ((size_t)pieces + n) * 4 + 16, false))) return rc;
        if ((rc = grow(ctx, ctx->gz_hcrc, ((size_t)n + 1) * 4 + 16, true))) return rc;
        if ((rc = grow(ctx, ctx->gz_windows, gzl::WIN * 4, false))) return rc;          // (never read: a member has no history before it)
        if ((rc = gz_text_room(ctx, f.carry, text_len))) return rc;
        if ((rc = gz_expand_tokens(ctx, ntok, tokcap, symcap))) return rc;
        if ((rc = gz_resolve_text(ctx, symcap, d_toff, n, f.carry, text_len, pieces))) return rc;
        uint32_t *d_flag = (uint32_t *)ctx->gz_crc.p + pieces;
        gzd::MemberCrcArgs ca;
        ca.syms = (const uint16_t *)ctx->gz_sym2.p;
        ca.stride = symcap;
        ca.lens = (const uint32_t *)ctx->gz_lens.p;
        ca.n = n;
        ca.crc = d_flag + 1;
        ca.table = (const uint32_t *)((uint8_t *)ctx->gz_tabs.p + 512);
        for (int j = 0; j < 5; j++) ca.op[j] = (uint32_t)crc32_combine_gen((z_off_t)(2048u << j));
        gzd::gz_member_crc<<<(n + 7) / 8, 256, 0, ctx->stream>>>(ca);
        CK(cudaGetLastError());
        ctx->launches += 2;                  // gz_member_crc and gz_decode: a round that stops before its text kernels counts none
        uint32_t *h = (uint32_t *)ctx->gz_hcrc.p;                                       // [0] the high-bit flag, [1..n] the members' CRCs
        CK(cudaMemcpyAsync(h, d_flag, ((size_t)n + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (uint32_t k = 0; k < n; k++)
            if (h[1 + k] != mem[k].crc) return fail(ctx, TDG_ERR_GZIP, std::string("gzip error in ") + f.path + ": corrupt BGZF member");
        if ((rc = gz_check_utf8(f, h[0], text_len))) return rc;
        if ((rc = f.to_sink(text_len))) return rc;
    } else {
        ctx->launches++;                                                                 // gz_decode
    }
    f.delivered += text_len;
    f.off = end;
    f.done = f.off == map.n;
    f.stats.rounds++;
    f.stats.chunks += n;
    f.stats.accepted += n;
    f.stats.ms_decode += gz_ms(t0, t1);
    f.stats.ms_resolve += gz_ms(t1, GzClock::now());
    if (f.debug)
        fprintf(stderr, "gzdev BGZF round: %u members, %zu compressed bytes, %llu bytes of text; upload + decode %.1f, rest %.1f ms\n", n, nb,
                (unsigned long long)text_len, gz_ms(t0, t1), gz_ms(t1, GzClock::now()));
    return TDG_OK;
}

// A round of an ordinary gzip stream: plan -> upload (or the bytes read ahead in the round before) -> scan ->
// decode -> which chunks continue the stream (chain) -> the text stage, with the windows passes and the CRC of
// the text, which st.advance holds against the member's trailer.
int gz_stream_round(GzFeed &f)
{
    using namespace tdg;
    tdg_ctx *ctx = f.ctx;
    gzc::Stream &st = f.st;
    const size_t file_n = f.map.n;
    const uint32_t max_chunks = std::min<uint32_t>(f.max_chunks, 65000);             // gz_ptr_*: a chunk index has 16 bits
    uint8_t *d_tabs = (uint8_t *)ctx->gz_tabs.p;
    uint8_t *d_window = d_tabs + 512 + 1024;
    int rc;
    // Chunk size, chosen per round from what is left of the file: every lane gets work when there is enough of
    // it, in steps of 16 KiB between 32 and 128 KiB (a chunk should hold a block start: zlib's blocks are
    // 10 - 30 KB of compressed data).  What a lane may produce: symbols up to 8 x its chunk (and room for a
    // large block), token slots up to 3 x its chunk (literal codes of 4 bits and more: two slots per compressed
    // byte); a chunk that needs more ends the device feed (the host reader takes over).
    size_t chunk = f.fixed_chunk;
    if (!chunk) {
        const size_t left = file_n - (size_t)(st.pos_bit >> 3);
        chunk = round_up((left + max_chunks - 1) / max_chunks, (size_t)16 << 10);
        chunk = std::min<size_t>(std::max<size_t>(chunk, (size_t)32 << 10), (size_t)128 << 10);
    }
    const uint32_t symcap = f.fixed_cap ? f.fixed_cap : (uint32_t)std::max<size_t>(8 * chunk, (size_t)256 << 10);
    const uint32_t tokcap = f.fixed_cap ? f.fixed_cap : (uint32_t)std::max<size_t>(3 * chunk, (size_t)128 << 10);
    const gzc::Round r = st.plan(chunk, max_chunks);
    const size_t nb = r.buf_end - r.buf_off;
    // ---- the round's compressed bytes: file -> pinned pieces -> device (or already there: see below)
    auto t0 = GzClock::now();
    const bool prefetched = f.pre_valid && f.pre_off <= r.buf_off && f.pre_end >= r.buf_end && (r.buf_off - f.pre_off) % 16 == 0;
    size_t comp_skip = 0;                                // where the round's bytes begin in the buffer
    if (prefetched) {
        f.cur ^= 1;                                      // the bytes sit in the other buffer: wait for their copies
        comp_skip = r.buf_off - f.pre_off;
        CK(cudaStreamWaitEvent(ctx->stream, ctx->gz_pre, 0));
    } else {
        rc = f.upload(f.cur, r.buf_off, r.buf_end, ctx->stream);
        if (rc) return rc;
    }
    f.pre_valid = false;
    Buf &comp = f.cur ? ctx->gz_comp2 : ctx->gz_comp;
    if ((rc = grow(ctx, ctx->gz_syms, (size_t)r.nchunks * tokcap * 2, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_meta, (size_t)r.nchunks * sizeof(gzl::Meta), false))) return rc;
    if ((rc = grow(ctx, ctx->gz_cand, (size_t)r.nchunks * gzd::MAXC * 4, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_ncand, (size_t)r.nchunks * 4, false))) return rc;
    if ((rc = grow(ctx, ctx->gz_hmeta, (size_t)r.nchunks * sizeof(gzl::Meta), true))) return rc;
    if ((rc = grow(ctx, ctx->gz_cold, (size_t)(r.nchunks + 8) * gzl::COLD_U16 * 2, false))) return rc;
    if (f.debug) CK(cudaStreamSynchronize(ctx->stream));
    auto t1 = GzClock::now();
    // ---- scan + decode
    gzd::RoundArgs a = gz_round_args(ctx, (const uint8_t *)comp.p + comp_skip, nb, r.nchunks, symcap, tokcap);      // (m_start / m_end stay null: this is one stream, not BGZF members)
    a.chunk_bytes = chunk;
    a.file_left = file_n - r.grid;
    a.pos_rel = r.pos_bit - (uint64_t)r.grid * 8;
    a.base_bit = (uint64_t)r.grid * 8;
    a.hist = r.hist;
    a.cand = (uint32_t *)ctx->gz_cand.p;
    a.ncand = (uint32_t *)ctx->gz_ncand.p;
    a.kraft3 = d_tabs;
    CK(cudaMemsetAsync(ctx->gz_ncand.p, 0, (size_t)r.nchunks * 4, ctx->stream));
    if (r.nchunks > 1) {
        const unsigned g = (r.nchunks - 1 + gzd::SCAN_WARPS - 1) / gzd::SCAN_WARPS;
        gzd::gz_scan<<<g, gzd::SCAN_WARPS * 32, gzd::SCAN_SMEM, ctx->stream>>>(a);
        CK(cudaGetLastError());
        ctx->launches++;
    }
    if (f.debug) CK(cudaStreamSynchronize(ctx->stream));
    auto t2 = GzClock::now();
    gzd::gz_decode<<<(r.nchunks + gzd::DEC_THREADS - 1) / gzd::DEC_THREADS, gzd::DEC_THREADS, gzd::DEC_SMEM, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    gzl::Meta *meta = (gzl::Meta *)ctx->gz_hmeta.p;
    CK(cudaMemcpyAsync(meta, ctx->gz_meta.p, (size_t)r.nchunks * sizeof(gzl::Meta), cudaMemcpyDeviceToHost, ctx->stream));
    // While the lanes inflate, this thread reads the bytes the NEXT round will most likely ask
    // for (every chunk accepted: its grid starts where this one's ends) and sends them to the
    // other buffer on the copy stream.
    double ms_prefetch = 0;
    const auto tp0 = GzClock::now();
    if (r.grid + (size_t)r.nchunks * chunk < file_n && r.nchunks == max_chunks) {
        f.pre_off = r.grid + (size_t)r.nchunks * chunk;  // (the next round's grid starts here or, with smaller chunks, a little further on)
        f.pre_end = std::min(file_n, f.pre_off + ((size_t)max_chunks + 2) * chunk);
        rc = f.upload(f.cur ^ 1, f.pre_off, f.pre_end, ctx->copy_stream);
        if (rc) return rc;
        CK(cudaEventRecord(ctx->gz_pre, ctx->copy_stream));
        f.pre_valid = true;
        ms_prefetch = gz_ms(tp0, GzClock::now());
    }
    CK(cudaStreamSynchronize(ctx->stream));
    auto t3 = GzClock::now();
    // ---- which chunks continue the stream
    const gzc::Outcome o = st.chain(r, meta, symcap);
    uint64_t text_len = o.text_off.back();
    uint32_t text_crc = 0;
    auto t4 = t3, t5 = t3;
    if (o.accepted && text_len) {
        const int go = f.sink.may_take(ctx, (size_t)text_len);
        if (go < 0) return go;
        if (go == 0) return TDG_STOP_ROUND;
        const uint32_t pieces = (uint32_t)((text_len + gzd::PIECE - 1) / gzd::PIECE);
        if ((rc = grow(ctx, ctx->gz_windows, ((size_t)o.accepted + 1) * (gzl::WIN * 4 + 1), false))) return rc;
        if ((rc = grow(ctx, ctx->gz_lens, (size_t)o.accepted * 4, false))) return rc;
        if ((rc = grow(ctx, ctx->gz_offs, ((size_t)o.accepted + 1) * 8, false))) return rc;
        if ((rc = grow(ctx, ctx->gz_crc, ((size_t)pieces + pieces / 256 + 2) * 4 + 16, false))) return rc;
        if ((rc = grow(ctx, ctx->gz_hcrc, ((size_t)pieces / 256 + 4) * 4 + 16, true))) return rc;
        if ((rc = gz_text_room(ctx, f.carry, text_len))) return rc;
        CK(cudaMemcpyAsync(ctx->gz_lens.p, o.lens.data(), o.lens.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        // tokens -> symbols (accepted chunks only)
        // the symbols: as many per chunk as the largest accepted chunk has
        uint32_t stride = 64;
        for (uint32_t len : o.lens) stride = std::max(stride, len);
        stride = (stride + 63u) & ~63u;
        if ((rc = grow(ctx, ctx->gz_sym2, (size_t)o.accepted * stride * 2, false))) return rc;
        if ((rc = grow(ctx, ctx->gz_ntok, (size_t)o.accepted * 4, false))) return rc;
        std::vector<uint32_t> ntok(o.accepted);
        for (uint32_t k = 0; k < o.accepted; k++) ntok[k] = o.lens[k] ? meta[k].ntok : 0u;
        for (const gzc::Repair &rp : o.repairs) ntok[rp.chunk] = 0;          // the host made these chunks' symbols
        if ((rc = gz_expand_tokens(ctx, ntok, tokcap, stride))) return rc;
        for (const gzc::Repair &rp : o.repairs)
            if (!rp.syms.empty())
                CK(cudaMemcpyAsync((uint16_t *)ctx->gz_sym2.p + (size_t)rp.chunk * stride, rp.syms.data(), rp.syms.size() * 2,
                                   cudaMemcpyHostToDevice, ctx->stream));
        if (f.debug) {
            CK(cudaStreamSynchronize(ctx->stream));
            fprintf(stderr, "gzdev expand: %.1f ms, %zu chunks made by the host\n", gz_ms(t3, GzClock::now()), o.repairs.size());
        }
        CK(cudaMemcpyAsync(ctx->gz_offs.p, o.text_off.data(), o.text_off.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        gzd::WinArgs w;
        w.syms = (const uint16_t *)ctx->gz_sym2.p;
        w.symcap = stride;
        w.out_len = (const uint32_t *)ctx->gz_lens.p;
        w.accepted = o.accepted;
        w.window_in = d_window;
        w.ptrs = (uint32_t *)ctx->gz_windows.p;
        w.done = (uint8_t *)ctx->gz_windows.p + ((size_t)o.accepted + 1) * gzl::WIN * 4;
        w.window_out = d_window;
        gzd::gz_ptr_init<<<o.accepted + 1, gzd::WIN_THREADS, 0, ctx->stream>>>(w);
        CK(cudaGetLastError());
        uint32_t passes = 1;
        while ((1u << (passes - 1)) < o.accepted + 1) passes++;          // chains are at most accepted + 1 long
        for (uint32_t ps = 0; ps < passes; ps++) gzd::gz_ptr_jump<<<o.accepted, gzd::WIN_THREADS, 0, ctx->stream>>>(w);
        CK(cudaGetLastError());
        ctx->launches += 1 + passes;
        if (f.debug) {
            CK(cudaStreamSynchronize(ctx->stream));
            fprintf(stderr, "gzdev windows: %u passes, %.1f ms\n", passes, gz_ms(t3, GzClock::now()));
        }
        if ((rc = gz_resolve_text(ctx, stride, (const uint64_t *)ctx->gz_offs.p, o.accepted, f.carry, text_len, pieces))) return rc;
        // the window behind the last accepted chunk opens the next round
        gzd::gz_ptr_take<<<8, gzd::WIN_THREADS, 0, ctx->stream>>>(w);
        CK(cudaGetLastError());
        ctx->launches++;
        // the pieces' raw CRCs: 256 full pieces fold into one on the device, the host folds the rest
        uint32_t *d_flag = (uint32_t *)ctx->gz_crc.p + pieces;
        const uint32_t nfull = (uint32_t)(text_len / gzd::PIECE), groups = (nfull + 255) / 256;
        uint32_t *d_group = d_flag + 1;
        if (groups) {
            gzd::CrcFoldArgs fa;
            fa.piece = (const uint32_t *)ctx->gz_crc.p;
            fa.nfull = nfull;
            fa.group = d_group;
            for (int j = 0; j < 8; j++) fa.op[j] = (uint32_t)crc32_combine_gen((z_off_t)((uint64_t)gzd::PIECE << j));
            gzd::gz_crc_fold<<<groups, 256, 0, ctx->stream>>>(fa);
            CK(cudaGetLastError());
            ctx->launches++;
        }
        // host copy: [0] the high-bit flag, [1 .. groups] the group CRCs, [groups + 1] the last (partial) piece's
        uint32_t *hcrc = (uint32_t *)ctx->gz_hcrc.p;
        CK(cudaMemcpyAsync(hcrc, d_flag, ((size_t)groups + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (pieces > nfull)
            CK(cudaMemcpyAsync(hcrc + groups + 1, (uint32_t *)ctx->gz_crc.p + nfull, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        t4 = GzClock::now();
        // CRC-32 of the round's text from the raw CRCs
        uLong raw = 0;
        if (groups) {
            const uLong op_group = crc32_combine_gen((z_off_t)((uint64_t)gzd::PIECE * 256));
            for (uint32_t g = 0; g + 1 < groups; g++) raw = crc32_combine_op(raw, hcrc[1 + g], op_group);
            const uint64_t last_group = (uint64_t)(nfull - (groups - 1) * 256u) * gzd::PIECE;
            raw = crc32_combine_op(raw, hcrc[groups], crc32_combine_gen((z_off_t)last_group));
        }
        if (pieces > nfull) raw = crc32_combine_op(raw, hcrc[groups + 1], crc32_combine_gen((z_off_t)(text_len - (uint64_t)nfull * gzd::PIECE)));
        text_crc = (uint32_t)(raw ^ crc32_combine_op(0xFFFFFFFFul, 0, crc32_combine_gen((z_off_t)text_len)) ^ 0xFFFFFFFFul);
        if ((rc = gz_check_utf8(f, hcrc[0], text_len))) return rc;
        t5 = GzClock::now();
    }
    if (!st.advance(r, o, text_len, text_crc))
        return fail(ctx, TDG_ERR_GZIP, std::string("gzip error in ") + f.path + ": incorrect data check");
    if (o.accepted && text_len && (rc = f.to_sink(text_len))) return rc;
    auto t6 = GzClock::now();
    f.done = st.eof;
    f.handover = st.handover;
    f.stats.rounds++;
    f.stats.chunks += r.nchunks;
    f.stats.accepted += o.accepted;
    f.stats.ms_upload += gz_ms(t0, t1);
    f.stats.ms_scan += gz_ms(t1, t2);
    f.stats.ms_decode += gz_ms(t2, t3);
    f.stats.ms_host += gz_ms(t4, t5);
    f.stats.ms_resolve += gz_ms(t3, t4);
    f.stats.ms_sink += gz_ms(t5, t6);
    if (f.debug)
        fprintf(stderr, "gzdev round: %u chunks of %zu KiB, %u accepted, %llu bytes of text; upload %.1f%s scan %.1f decode %.1f "
                        "(host read the next round's bytes meanwhile: %.1f) expand+windows+resolve %.1f crc/utf8 %.1f sink %.1f ms%s%s\n",
                r.nchunks, chunk >> 10, o.accepted, (unsigned long long)text_len, gz_ms(t0, t1), prefetched ? " (prefetched)" : "", gz_ms(t1, t2),
                gz_ms(t2, t3), ms_prefetch, gz_ms(t3, t4), gz_ms(t4, t5),
                gz_ms(t5, t6), st.handover ? "  -> host reader: " : "", st.handover ? st.why : "");
    return TDG_OK;
}

// Inflates `path` (an ordinary gzip file or BGZF) on the device round by round and hands every round's
// text to `sink`.  handled = false: nothing was done (a header this feed does not take: the host
// feeder starts from the beginning).  Otherwise the text went to the sink up to the end of the
// file, or up to the place `ho` describes (ho.active), where the host feeder continues.
int gz_device_feed(tdg_ctx *ctx, const char *path, GzSink &sink, bool &handled, GzHandover &ho, size_t &carry, GzStats &stats,
                   tdg::Utf8State *u8)
{
    using namespace tdg;
    handled = false;
    ho = GzHandover();
    GzFeed f{ctx, path, sink, carry, stats, u8};
    GzMap &map = f.map;
    map.fd = ::open(path, O_RDONLY);
    if (map.fd < 0) return TDG_OK;                       // the host feeder reports it
    struct stat sb;
    if (fstat(map.fd, &sb) != 0 || !S_ISREG(sb.st_mode) || sb.st_size < 32) return TDG_OK;
    map.n = (size_t)sb.st_size;
    void *mp = mmap(nullptr, map.n, PROT_READ, MAP_PRIVATE, map.fd, 0);
    if (mp == MAP_FAILED) return TDG_OK;
    map.p = (const uint8_t *)mp;
    const bool bgzf = Feeder::is_bgzf(map.p, std::min<size_t>(map.n, 1024));
    if (!bgzf && !f.st.open(map.p, map.n)) return TDG_OK;
    int rc = gz_tables(ctx);
    if (rc) return rc;
    rc = ensure_slots(ctx);
    if (rc) return rc;
    f.max_chunks = (uint32_t)ctx->sm_count * gzd::DEC_THREADS;          // one lane per chunk (or member), one CTA per SM
    if (const char *e = getenv("TDG_GZDEV_MAXCHUNKS")) f.max_chunks = (uint32_t)std::max(1, atoi(e));
    if (const char *e = getenv("TDG_GZDEV_CHUNK")) f.fixed_chunk = std::max<size_t>(4096, strtoull(e, nullptr, 10) / 16 * 16);
    if (const char *e = getenv("TDG_GZDEV_SYMCAP")) f.fixed_cap = (uint32_t)std::max<unsigned long long>(1024, strtoull(e, nullptr, 10));
    f.debug = getenv("TDG_GZDEV_DEBUG") != nullptr;
    f.threads = gz_io_threads();
    uint8_t *d_window = (uint8_t *)ctx->gz_tabs.p + 512 + 1024;
    if (!bgzf) CK(cudaMemsetAsync(d_window, 0, gzl::WIN, ctx->stream));      // a stream has no history in front of it
    handled = true;
    carry = 0;

    const int oom_round = getenv("TDG_GZDEV_OOM_ROUND") ? atoi(getenv("TDG_GZDEV_OOM_ROUND")) : -1;      // test hook
    int (*round)(GzFeed &) = bgzf ? gz_bgzf_round : gz_stream_round;
    for (int round_no = 0; !f.done && !f.handover; round_no++) {
        f.sunk = false;
        rc = round_no == oom_round ? fail(ctx, TDG_ERR_NOMEM, "buffer of 0 bytes: simulated (TDG_GZDEV_OOM_ROUND)") : round(f);
        if (!f.sunk && (rc == TDG_ERR_NOMEM || rc == TDG_STOP_ROUND)) f.handover = true;         // at the state the round began in
        else if (rc) return rc;
    }
    if (f.handover) {
        ho.active = true;
        ho.bgzf = bgzf;
        ho.bgzf_off = f.off;
        ho.to_zlib = f.st.to_zlib;
        ho.pos_bit = f.st.pos_bit;
        ho.hist = f.st.hist;
        ho.crc = f.st.crc;
        ho.member_len = f.st.member_len;
        ho.delivered = bgzf ? f.delivered : f.st.delivered;
        if (!bgzf) {
            ho.window.resize(gzl::WIN);
            CK(cudaMemcpyAsync(ho.window.data(), d_window, gzl::WIN, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
        }
    }
    return TDG_OK;
}

// tdg_count_file's sink: whole lines go to the counting kernel, the rest is carried
struct GzCountSink : GzSink {
    uint64_t reads_limit;
    LimitState *lim;
    GzCountSink(uint64_t limit, LimitState *l) : reads_limit(limit), lim(l) {}
    int may_take(tdg_ctx *ctx, size_t len) override { return lim ? limit_admits(ctx, *lim, len) : 1; }
    int text(tdg_ctx *ctx, uint8_t *d_buf, size_t &carry, size_t len) override
    {
        const size_t total = carry + len;
        // the last line end: look at the tail on the host
        size_t cut = 0;
        for (size_t tail = std::min<size_t>(total, (size_t)1 << 20);; tail = std::min(total, tail * 8)) {
            int rc = grow(ctx, ctx->gz_htail, tail, true);
            if (rc) return rc;
            CK(cudaMemcpyAsync(ctx->gz_htail.p, d_buf + (total - tail), tail, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            const size_t c = line_cut((const uint8_t *)ctx->gz_htail.p, tail);
            if (c) { cut = total - tail + c; break; }
            if (tail == total) break;
        }
        if (cut) {
            int rc = launch_chunk<true>(ctx, d_buf, cut, TDG_LINE_CHAINED, 0, reads_limit);
            if (rc) return rc;
        }
        const size_t rest = total - cut;
        if (rest && cut) {
            int rc = grow(ctx, ctx->gz_carry, rest, false);
            if (rc) return rc;
            CK(cudaMemcpyAsync(ctx->gz_carry.p, d_buf + cut, rest, cudaMemcpyDeviceToDevice, ctx->stream));
            CK(cudaMemcpyAsync(d_buf, ctx->gz_carry.p, rest, cudaMemcpyDeviceToDevice, ctx->stream));
        }
        carry = rest;
        return TDG_OK;
    }
};

// tdg_gz_inflate_host's sink: the text goes to a host buffer
struct GzCopySink : GzSink {
    uint8_t *dst;
    size_t cap, used = 0;
    GzCopySink(uint8_t *d, size_t c) : dst(d), cap(c) {}
    int text(tdg_ctx *ctx, uint8_t *d_buf, size_t &carry, size_t len) override
    {
        if (used + len > cap) return fail(ctx, TDG_ERR_ARG, "output buffer too small");
        CK(cudaMemcpyAsync(dst + used, d_buf + carry, len, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        used += len;
        carry = 0;
        return TDG_OK;
    }
};

bool gz_device_wanted(const tdg_ctx *ctx, const char *path, uint64_t reads_limit)
{
    if (const char *e = getenv("TDG_GZDEV")) {
        if (atoi(e) == 0) return false;
    }
    // a maxreads whose line can lie in the first piece (LimitState::init): the reader stops early, small host pieces
    if (reads_limit < ((uint64_t)1 << 60) && 4 * reads_limit <= (uint64_t)ctx->chunk_bytes + 2) return false;
    uint64_t min_size = (uint64_t)8 << 20;
    if (const char *e = getenv("TDG_GZDEV_MIN")) min_size = strtoull(e, nullptr, 10);
    struct stat sb;
    return stat(path, &sb) == 0 && S_ISREG(sb.st_mode) && (uint64_t)sb.st_size >= min_size;
}

