// BGZF writer of the barcode splitter (sm_100a): every barcode's output stream is cut into members of
// 65,280 bytes (bgzip's block size), and each member becomes one gzip member with the `BC` extra
// field -- an independent deflate stream, compressed by one CTA.
//
// Kernels, in launch order (the host plans the members, tdg_api.cu: bgzf_run):
//   bgzf_deflate   one CTA per member, the member in shared memory:
//                    matches   windows of 256 positions; a position looks up the positions of
//                              earlier windows in hash tables (4-byte hash: two ways, 8-byte hash:
//                              one way), length <= 258, distance <= 32,768, all inside the member
//                    parse     greedy: token starts = the path 0 -> 0 + max(1, len[0]) -> ...; every
//                              thread walks its 255-byte segment, one thread then joins the walks
//                    codes     literal/length and distance histograms, length-limited Huffman codes
//                              (<= 15 bits; the code-length code <= 7 bits), one thread per tree
//                    bits      token bit offsets from a block-wide scan; bits OR-ed into the slot
//                    member    min(dynamic block, stored block), CRC-32 of the shared-memory copy
//                              (the operator tree of tdg_gzdev.cuh), header and trailer
//   tile_scan      (tdg_split.cuh) exclusive prefix over the member sizes
//   bgzf_pack      the members end to end, in barcode order
//   bgzf_copy      the barcodes' new pending tails
//
// Rules the output keeps, so that zlib, Python's gzip, tdg_pgz.h and the device feed's member mode all
// take it: codes are complete (never over-subscribed or incomplete), every tree has at least two
// codes, symbols 286/287 and distances 30/31 never occur, HLIT >= 257, HDIST >= 1, HCLEN >= 4, repeat
// code 16 never starts the literal/length or the distance lengths, Huffman codes are sent bit-reversed.
//
// The phases are plain functions of (shared state, thread index) so that a CPU harness
// (tests/native/bgzf_check.cpp) can run them one thread after the other and hold them to zlib.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#include "tdg_gzdev.cuh"
#define BZ_HD __host__ __device__
#else
#define BZ_HD
#endif

namespace tdg {
namespace bz {

constexpr uint32_t BLOCK = 65280;               // bytes of a full member (bgzip's BGZF_BLOCK_SIZE)
constexpr uint32_t THREADS = 256;
constexpr uint32_t SEG = BLOCK / THREADS;       // 255: bytes of a thread's segment (parse, bits, CRC)
constexpr uint32_t NLIT = 286, NDIST = 30, NCL = 19, NSYM = NLIT + NDIST + NCL;
constexpr uint32_t T4_BITS = 11, T4_N = 1u << T4_BITS;
constexpr uint32_t T8_BITS = 12, T8_N = 1u << T8_BITS;
constexpr uint32_t TAB_WORDS = 2 * T4_N + T8_N;
constexpr uint32_t MARK_WORDS = (BLOCK + 31) / 32;
constexpr uint32_t HEAD_BYTES = 18, TRAIL_BYTES = 8;
constexpr uint32_t SLOT_EXTRA = 64;             // a member's slot: its input size + this, rounded to 16
constexpr uint32_t EOF_BYTES = 28;
static_assert(SEG * THREADS == BLOCK, "a member is 256 segments");
static_assert(2 * (NLIT + NDIST) <= TAB_WORDS, "the trees' sort scratch fits the table space");

// the 28-byte end-of-file member of the BGZF specification (SAMv1 4.1.2)
BZ_HD inline uint8_t eof_byte(uint32_t i)
{
    const uint8_t head[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0};
    if (i < 16) return head[i];
    if (i == 16) return 0x1b;
    if (i == 18) return 3;
    return 0;
}

struct Shared {                                  // one CTA's shared memory
    uint8_t in[BLOCK + 16];                      // the member (+ zero padding for the hashes)
    uint32_t tab[TAB_WORDS];                     // matching: t4 way 0, t4 way 1, t8 (positions + 1); then sort scratch
    uint32_t mark[MARK_WORDS];                   // token starts
    uint32_t freq[NSYM];                         // literal/length, distance, code-length frequencies
    uint16_t code[NSYM];                         // bit-reversed codes
    uint8_t len[NSYM + 1];                       // code lengths
    uint16_t rle[NLIT + NDIST];                  // code-length symbols: sym | extra << 5
    uint32_t seg[THREADS];                       // per segment: exit of the walk, then bits, then bit offset
    uint32_t crc[THREADS];
    uint32_t nrle, hlit, hdist, hclen, head_bits, total_bits, dynamic;
};

struct Job {                                     // one member
    const uint8_t *src0;                         // first part (a barcode's pending tail)
    uint32_t len0;
    const uint8_t *src1;                         // second part (new bytes)
    uint32_t len1;
    uint32_t n;                                  // len0 + len1 <= BLOCK
    uint32_t *m;                                 // [n] per position: len << 16 | (dist - 1), 0 = literal
    uint8_t *out;                                // the member's slot (16-byte aligned, zeroed by phase_load)
};

// ---- atomics that the CPU harness runs as plain operations
BZ_HD inline uint32_t at_max(uint32_t *p, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return atomicMax(p, v);
#else
    const uint32_t o = *p;
    if (v > o) *p = v;
    return o;
#endif
}
BZ_HD inline void at_or(uint32_t *p, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    atomicOr(p, v);
#else
    *p |= v;
#endif
}
BZ_HD inline void at_add(uint32_t *p, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
BZ_HD inline uint32_t msb(uint32_t x)          // x > 0
{
#if defined(__CUDA_ARCH__)
    return 31u - __clz(x);
#else
    return 31u - (uint32_t)__builtin_clz(x);
#endif
}

// ---- symbols of RFC 1951 3.2.5
BZ_HD inline void len_sym(uint32_t l, uint32_t &sym, uint32_t &nx, uint32_t &x)     // 3 <= l <= 258
{
    const uint32_t v = l - 3;
    if (l == 258) { sym = 285; nx = 0; x = 0; }
    else if (v < 8) { sym = 257 + v; nx = 0; x = 0; }
    else {
        const uint32_t b = msb(v);
        sym = 257 + 4 * (b - 1) + ((v >> (b - 2)) & 3u);
        nx = b - 2;
        x = v & ((1u << nx) - 1u);
    }
}
BZ_HD inline void dist_sym(uint32_t d, uint32_t &sym, uint32_t &nx, uint32_t &x)    // 1 <= d <= 32768
{
    const uint32_t v = d - 1;
    if (v < 4) { sym = v; nx = 0; x = 0; }
    else {
        const uint32_t b = msb(v);
        sym = 2 * b + ((v >> (b - 1)) & 1u);
        nx = b - 1;
        x = v & ((1u << nx) - 1u);
    }
}

// ---- Huffman code lengths
// Moffat & Katajainen, "In-place calculation of minimum-redundancy codes" (1995): A[0..n) holds the
// frequencies in ascending order and receives the code lengths (A[0] the longest).
BZ_HD inline void min_redundancy(uint32_t *A, int n)
{
    if (n == 0) return;
    if (n == 1) { A[0] = 1; return; }
    A[0] += A[1];
    int root = 0, leaf = 2, next;
    for (next = 1; next < n - 1; next++) {
        if (leaf >= n || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = (uint32_t)next; }
        else A[next] = A[leaf++];
        if (leaf >= n || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = (uint32_t)next; }
        else A[next] += A[leaf++];
    }
    A[n - 2] = 0;
    for (next = n - 3; next >= 0; next--) A[next] = A[A[next]] + 1;
    int avbl = 1, used = 0, dpth = 0;
    root = n - 2;
    next = n - 1;
    while (avbl > 0) {
        while (root >= 0 && (int)A[root] == dpth) { used++; root--; }
        while (avbl > used) { A[next--] = (uint32_t)dpth; avbl--; }
        avbl = 2 * used;
        dpth++;
        used = 0;
    }
}

// Code lengths <= maxbits for freq[0..n), complete, with at least two codes (an unused symbol of
// the lowest index joins with count 1 when fewer are used: zlib's build_tree does the same).
// freq is updated accordingly.  scratch: 2 * n words.  The frequencies must sum below 2^32.
BZ_HD inline void huff_lengths(uint32_t *freq, uint32_t n, uint32_t maxbits, uint8_t *len, uint32_t *scratch)
{
    uint32_t used = 0;
    for (uint32_t s = 0; s < n; s++) used += freq[s] != 0;
    for (uint32_t s = 0; s < n && used < 2; s++)
        if (!freq[s]) { freq[s] = 1; used++; }
    uint32_t *sym = scratch, *A = scratch + n;
    uint32_t m = 0;
    for (uint32_t s = 0; s < n; s++) {
        len[s] = 0;
        if (freq[s]) sym[m++] = s;
    }
    // shell sort by (frequency, symbol)
    for (uint32_t gap = m / 2; gap > 0; gap = gap == 2 ? 1 : gap * 5 / 11) {
        for (uint32_t i = gap; i < m; i++) {
            const uint32_t t = sym[i];
            uint32_t j = i;
            while (j >= gap && (freq[sym[j - gap]] > freq[t] || (freq[sym[j - gap]] == freq[t] && sym[j - gap] > t))) {
                sym[j] = sym[j - gap];
                j -= gap;
            }
            sym[j] = t;
        }
    }
    for (uint32_t i = 0; i < m; i++) A[i] = freq[sym[i]];
    min_redundancy(A, (int)m);
    uint32_t count[33];
    for (uint32_t b = 0; b <= 32; b++) count[b] = 0;
    for (uint32_t i = 0; i < m; i++) count[A[i] < 32 ? A[i] : 32]++;
    // lengths above maxbits become maxbits; then codes move down until the Kraft sum is exactly 1
    for (uint32_t b = maxbits + 1; b <= 32; b++) { count[maxbits] += count[b]; count[b] = 0; }
    uint32_t total = 0;
    for (uint32_t b = maxbits; b > 0; b--) total += count[b] << (maxbits - b);
    while (total != (1u << maxbits)) {
        count[maxbits]--;
        for (uint32_t b = maxbits - 1; b > 0; b--)
            if (count[b]) { count[b]--; count[b + 1] += 2; break; }
        total--;
    }
    uint32_t j = m;                              // the most frequent symbols get the shortest codes
    for (uint32_t b = 1; b <= maxbits; b++)
        for (uint32_t k = count[b]; k > 0; k--) len[sym[--j]] = (uint8_t)b;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first stream
BZ_HD inline void huff_codes(const uint8_t *len, uint32_t n, uint16_t *code)
{
    uint32_t cnt[16], next[16];
    for (uint32_t b = 0; b < 16; b++) cnt[b] = 0;
    for (uint32_t s = 0; s < n; s++) cnt[len[s]]++;
    cnt[0] = 0;
    uint32_t c = 0;
    next[0] = 0;
    for (uint32_t b = 1; b < 16; b++) {
        c = (c + cnt[b - 1]) << 1;
        next[b] = c;
    }
    for (uint32_t s = 0; s < n; s++) {
        const uint32_t l = len[s];
        if (!l) { code[s] = 0; continue; }
        uint32_t v = next[l]++, r = 0;
        for (uint32_t k = 0; k < l; k++) { r = (r << 1) | (v & 1u); v >>= 1; }
        code[s] = (uint16_t)r;
    }
}

// run-length code of lens[0..n) with the code-length alphabet (RFC 1951 3.2.7), appended at out[k..)
BZ_HD inline uint32_t rle_lengths(const uint8_t *lens, uint32_t n, uint16_t *out, uint32_t k)
{
    uint32_t i = 0;
    while (i < n) {
        const uint32_t v = lens[i];
        uint32_t run = 1;
        while (i + run < n && lens[i + run] == v) run++;
        i += run;
        if (v == 0) {
            while (run >= 3) {
                const uint32_t r = run >= 11 ? (run < 138 ? run : 138) : run;
                out[k++] = r >= 11 ? (uint16_t)(18 | (r - 11) << 5) : (uint16_t)(17 | (r - 3) << 5);
                run -= r;
            }
        } else {
            out[k++] = (uint16_t)v;
            run--;
            while (run >= 3) {
                const uint32_t r = run < 6 ? run : 6;
                out[k++] = (uint16_t)(16 | (r - 3) << 5);
                run -= r;
            }
        }
        while (run > 0) { out[k++] = (uint16_t)v; run--; }
    }
    return k;
}

BZ_HD inline uint32_t cl_extra_bits(uint32_t sym) { return sym == 16 ? 2u : sym == 17 ? 3u : sym == 18 ? 7u : 0u; }

BZ_HD inline uint32_t cl_order(uint32_t i)      // the order in which the code-length code's lengths are sent
{
    const uint8_t order[NCL] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    return order[i];
}

// bits OR-ed into zeroed 32-bit words from an absolute bit position on
struct Bits {
    uint32_t *w;
    uint64_t acc;
    uint32_t nacc;
    BZ_HD Bits(uint32_t *words, uint32_t bitpos) : w(words + (bitpos >> 5)), acc(0), nacc(bitpos & 31u) {}
    BZ_HD void put(uint32_t v, uint32_t nb)     // nb <= 32, v < 2^nb
    {
        acc |= (uint64_t)v << nacc;
        nacc += nb;
        if (nacc >= 32) {
            at_or(w++, (uint32_t)acc);
            acc >>= 32;
            nacc -= 32;
        }
    }
    BZ_HD void flush()
    {
        if (nacc) at_or(w, (uint32_t)acc);
    }
};

BZ_HD inline uint32_t step(uint32_t m) { return m ? (m >> 16) : 1u; }
BZ_HD inline bool marked(const Shared &s, uint32_t p) { return (s.mark[p >> 5] >> (p & 31u)) & 1u; }
BZ_HD inline void clear_marks(Shared &s, uint32_t a, uint32_t b)
{
    while (a < b) {
        const uint32_t bit = a & 31u, cnt = (32u - bit) < (b - a) ? (32u - bit) : (b - a);
        const uint32_t mask = cnt == 32u ? 0xFFFFFFFFu : ((1u << cnt) - 1u) << bit;
        s.mark[a >> 5] &= ~mask;
        a += cnt;
    }
}
BZ_HD inline uint32_t hash4(const uint8_t *p)
{
    const uint32_t v = p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
    return (v * 2654435761u) >> (32 - T4_BITS);
}
BZ_HD inline uint32_t hash8(const uint8_t *p)
{
    const uint32_t a = p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
    const uint32_t b = p[4] | (uint32_t)p[5] << 8 | (uint32_t)p[6] << 16 | (uint32_t)p[7] << 24;
    return ((a * 2654435761u) ^ (b * 0x85EBCA77u)) >> (32 - T8_BITS);
}
BZ_HD inline uint32_t seg_end(uint32_t t, uint32_t n) { return (t + 1) * SEG < n ? (t + 1) * SEG : n; }

// ---- phases (each one ends in a barrier of the CTA)

// the member into shared memory; tables, histograms and marks cleared; the slot zeroed
BZ_HD inline void phase_load(Shared &s, const Job &j, uint32_t tid)
{
    for (uint32_t i = tid; i < j.n; i += THREADS) s.in[i] = i < j.len0 ? j.src0[i] : j.src1[i - j.len0];
    if (tid < 16) s.in[j.n + tid] = 0;
    for (uint32_t i = tid; i < TAB_WORDS; i += THREADS) s.tab[i] = 0;
    for (uint32_t i = tid; i < MARK_WORDS; i += THREADS) s.mark[i] = 0;
    for (uint32_t i = tid; i < NSYM; i += THREADS) s.freq[i] = i == 256 ? 1u : 0u;     // one end-of-block
    uint32_t *w = (uint32_t *)j.out;
    const uint32_t words = (j.n + SLOT_EXTRA) / 4;
    for (uint32_t i = tid; i < words; i += THREADS) w[i] = 0;
}

// longest match of position ws + tid against the positions of earlier windows
BZ_HD inline void phase_find(Shared &s, const Job &j, uint32_t ws, uint32_t tid)
{
    const uint32_t i = ws + tid;
    if (i >= j.n) return;
    uint32_t best = 0, bdist = 0;
    if (i + 4 <= j.n) {
        uint32_t cand[3];
        const uint32_t h4 = hash4(s.in + i);
        cand[0] = s.tab[h4];
        cand[1] = s.tab[T4_N + h4];
        cand[2] = i + 8 <= j.n ? s.tab[2 * T4_N + hash8(s.in + i)] : 0u;
        const uint32_t maxl = j.n - i < 258u ? j.n - i : 258u;
        for (int k = 0; k < 3; k++) {
            const uint32_t c = cand[k];
            if (!c || i - (c - 1) > 32768u || (k > 0 && c == cand[0]) || (k == 2 && c == cand[1])) continue;
            const uint8_t *a = s.in + (c - 1), *b = s.in + i;
            uint32_t l = 0;
            while (l < maxl && a[l] == b[l]) l++;
            if (l > best || (l == best && i - (c - 1) < bdist)) { best = l; bdist = i - (c - 1); }
        }
    }
    j.m[i] = best >= 4 ? (best << 16 | (bdist - 1)) : 0u;
}

// positions ws .. ws + 255 join the tables: way 0 of t4 keeps the latest position before the window
// being looked up, way 1 the one way 0 held before that window (the thread that meets the value from
// before this window moves it there: exactly one does)
BZ_HD inline void phase_insert(Shared &s, const Job &j, uint32_t ws, uint32_t tid)
{
    const uint32_t i = ws + tid;
    if (i + 4 > j.n) return;
    const uint32_t h4 = hash4(s.in + i);
    const uint32_t old = at_max(&s.tab[h4], i + 1);
    if (old <= ws) s.tab[T4_N + h4] = old;
    if (i + 8 <= j.n) at_max(&s.tab[2 * T4_N + hash8(s.in + i)], i + 1);
}

// the greedy parse inside the thread's segment, starting at the segment's first byte
BZ_HD inline void phase_walk(Shared &s, const Job &j, uint32_t tid)
{
    uint32_t p = tid * SEG;
    const uint32_t hi = seg_end(tid, j.n);
    while (p < hi) {
        at_or(&s.mark[p >> 5], 1u << (p & 31u));
        p += step(j.m[p]);
    }
    s.seg[tid] = p;
}

// one thread: the true path enters segment t at e; it follows its own steps until it meets a position
// the segment's walk took (from there on the two agree) or leaves the segment.  Marks the true path
// does not take are cleared.
BZ_HD inline void phase_join(Shared &s, const Job &j)
{
    uint32_t e = 0;
    for (uint32_t t = 0; t < THREADS && t * SEG < j.n; t++) {
        const uint32_t lo = t * SEG, hi = seg_end(t, j.n);
        if (e >= hi) { clear_marks(s, lo, hi); continue; }
        clear_marks(s, lo, e);
        uint32_t p = e;
        for (;;) {
            if (marked(s, p)) { e = s.seg[t]; break; }
            s.mark[p >> 5] |= 1u << (p & 31u);
            const uint32_t q = p + step(j.m[p]);
            clear_marks(s, p + 1, q < hi ? q : hi);
            if (q >= hi) { e = q; break; }
            p = q;
        }
    }
}

BZ_HD inline void phase_hist(Shared &s, const Job &j, uint32_t tid)
{
    const uint32_t hi = seg_end(tid, j.n);
    for (uint32_t p = tid * SEG; p < hi; p++) {
        if (!marked(s, p)) continue;
        const uint32_t m = j.m[p];
        if (m) {
            uint32_t sym, nx, x;
            len_sym(m >> 16, sym, nx, x);
            at_add(&s.freq[sym], 1);
            dist_sym((m & 0xFFFFu) + 1, sym, nx, x);
            at_add(&s.freq[NLIT + sym], 1);
        } else {
            at_add(&s.freq[s.in[p]], 1);
        }
    }
}

// which = 0: literal/length tree, 1: distance tree (two threads, side by side)
BZ_HD inline void phase_tree(Shared &s, uint32_t which)
{
    const uint32_t base = which ? NLIT : 0, n = which ? NDIST : NLIT;
    huff_lengths(s.freq + base, n, 15, s.len + base, s.tab + (which ? 2 * NLIT : 0));
    huff_codes(s.len + base, n, s.code + base);
}

// one thread: the code-length tree and the header's size
BZ_HD inline void phase_header(Shared &s)
{
    uint32_t hlit = NLIT, hdist = NDIST;
    while (hlit > 257 && !s.len[hlit - 1]) hlit--;
    while (hdist > 1 && !s.len[NLIT + hdist - 1]) hdist--;
    uint32_t k = rle_lengths(s.len, hlit, s.rle, 0);
    k = rle_lengths(s.len + NLIT, hdist, s.rle, k);
    uint32_t *cf = s.freq + NLIT + NDIST;
    uint8_t *cl = s.len + NLIT + NDIST;
    for (uint32_t c = 0; c < NCL; c++) cf[c] = 0;
    for (uint32_t i = 0; i < k; i++) cf[s.rle[i] & 31u]++;
    huff_lengths(cf, NCL, 7, cl, s.tab);
    huff_codes(cl, NCL, s.code + NLIT + NDIST);
    uint32_t hclen = NCL;
    while (hclen > 4 && !cl[cl_order(hclen - 1)]) hclen--;
    uint32_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
    for (uint32_t i = 0; i < k; i++) bits += cl[s.rle[i] & 31u] + cl_extra_bits(s.rle[i] & 31u);
    s.nrle = k;
    s.hlit = hlit;
    s.hdist = hdist;
    s.hclen = hclen;
    s.head_bits = bits;
}

BZ_HD inline uint32_t token_bits(const Shared &s, uint32_t m, uint8_t lit)
{
    if (!m) return s.len[lit];
    uint32_t sym, nx, x, bits;
    len_sym(m >> 16, sym, nx, x);
    bits = s.len[sym] + nx;
    dist_sym((m & 0xFFFFu) + 1, sym, nx, x);
    return bits + s.len[NLIT + sym] + nx;
}

BZ_HD inline void phase_seg_bits(Shared &s, const Job &j, uint32_t tid)
{
    const uint32_t hi = seg_end(tid, j.n);
    uint32_t bits = 0;
    for (uint32_t p = tid * SEG; p < hi; p++)
        if (marked(s, p)) bits += token_bits(s, j.m[p], s.in[p]);
    s.seg[tid] = bits;
}

// one thread: segment bit offsets, the block's size, dynamic or stored
BZ_HD inline void phase_scan(Shared &s, const Job &j)
{
    uint32_t run = s.head_bits;
    for (uint32_t t = 0; t < THREADS; t++) {
        const uint32_t b = s.seg[t];
        s.seg[t] = run;
        run += b;
    }
    s.total_bits = run + s.len[256];
    s.dynamic = (s.total_bits + 7) / 8 < j.n + 5 ? 1u : 0u;
}

BZ_HD inline uint32_t data_bytes(const Shared &s, const Job &j) { return s.dynamic ? (s.total_bits + 7) / 8 : j.n + 5; }

BZ_HD inline void phase_emit(Shared &s, const Job &j, uint32_t tid)
{
    uint8_t *data = j.out + HEAD_BYTES;
    if (!s.dynamic) {
        if (tid == 0) {
            data[0] = 1;                                            // BFINAL, BTYPE 00
            data[1] = (uint8_t)j.n;
            data[2] = (uint8_t)(j.n >> 8);
            data[3] = (uint8_t)~j.n;
            data[4] = (uint8_t)(~j.n >> 8);
        }
        for (uint32_t i = tid; i < j.n; i += THREADS) data[5 + i] = s.in[i];
        return;
    }
    uint32_t *words = (uint32_t *)j.out;
    const uint32_t base = HEAD_BYTES * 8;
    if (tid == 0) {
        Bits o(words, base);
        o.put(1 | 2 << 1, 3);                                       // BFINAL, BTYPE 10
        o.put(s.hlit - 257, 5);
        o.put(s.hdist - 1, 5);
        o.put(s.hclen - 4, 4);
        const uint8_t *cl = s.len + NLIT + NDIST;
        const uint16_t *cc = s.code + NLIT + NDIST;
        for (uint32_t i = 0; i < s.hclen; i++) o.put(cl[cl_order(i)], 3);
        for (uint32_t i = 0; i < s.nrle; i++) {
            const uint32_t sym = s.rle[i] & 31u;
            o.put(cc[sym], cl[sym]);
            if (sym >= 16) o.put(s.rle[i] >> 5, cl_extra_bits(sym));
        }
        o.flush();
        Bits e(words, base + s.total_bits - s.len[256]);
        e.put(s.code[256], s.len[256]);
        e.flush();
    }
    const uint32_t hi = seg_end(tid, j.n);
    Bits o(words, base + s.seg[tid]);
    for (uint32_t p = tid * SEG; p < hi; p++) {
        if (!marked(s, p)) continue;
        const uint32_t m = j.m[p];
        if (!m) { o.put(s.code[s.in[p]], s.len[s.in[p]]); continue; }
        uint32_t sym, nx, x;
        len_sym(m >> 16, sym, nx, x);
        o.put(s.code[sym] | x << s.len[sym], s.len[sym] + nx);
        dist_sym((m & 0xFFFFu) + 1, sym, nx, x);
        o.put(s.code[NLIT + sym] | x << s.len[NLIT + sym], s.len[NLIT + sym] + nx);
    }
    o.flush();
}

// gzip header with the BC field, and the trailer; returns the member's size
BZ_HD inline uint32_t write_frame(uint8_t *out, uint32_t data_len, uint32_t crc, uint32_t isize)
{
    const uint32_t size = HEAD_BYTES + data_len + TRAIL_BYTES;
    for (uint32_t i = 0; i < 16; i++) out[i] = eof_byte(i);
    out[16] = (uint8_t)(size - 1);
    out[17] = (uint8_t)((size - 1) >> 8);
    uint8_t *t = out + HEAD_BYTES + data_len;
    for (uint32_t i = 0; i < 4; i++) {
        t[i] = (uint8_t)(crc >> (8 * i));
        t[4 + i] = (uint8_t)(isize >> (8 * i));
    }
    return size;
}

#if defined(__CUDACC__)

struct Member {                      // host-planned
    const uint8_t *src0;
    const uint8_t *src1;
    uint32_t len0, len1;
    unsigned long long in_off;       // prefix of the members' sizes: the match array's offset
    unsigned long long slot;         // byte offset of the member's slot in `work`
};

struct DeflateArgs {
    const Member *mem;
    uint32_t n;
    uint32_t *match;                 // [sum of sizes]
    uint8_t *work;
    uint32_t *size;                  // [n + 1] member sizes (then scanned in place by tile_scan)
    const uint32_t *table;           // CRC-32 table (reflected polynomial)
    uint32_t op[8];                  // x^(8 * SEG * 2^j) modulo the polynomial
};

__global__ void __launch_bounds__(THREADS, 2) bgzf_deflate(const DeflateArgs a)
{
    extern __shared__ uint4 bz_smem[];
    Shared &s = *reinterpret_cast<Shared *>(bz_smem);
    const uint32_t tid = threadIdx.x;
    const Member d = a.mem[blockIdx.x];
    Job j;
    j.src0 = d.src0;
    j.len0 = d.len0;
    j.src1 = d.src1;
    j.len1 = d.len1;
    j.n = d.len0 + d.len1;
    j.m = a.match + d.in_off;
    j.out = a.work + d.slot;
    if (j.n == 0) {                                  // the end-of-file member
        if (tid < EOF_BYTES) j.out[tid] = eof_byte(tid);
        if (tid == 0) a.size[blockIdx.x] = EOF_BYTES;
        return;
    }
    phase_load(s, j, tid);
    __syncthreads();
    for (uint32_t ws = 0; ws < j.n; ws += THREADS) {
        phase_find(s, j, ws, tid);
        __syncthreads();
        phase_insert(s, j, ws, tid);
        __syncthreads();
    }
    phase_walk(s, j, tid);
    __syncthreads();
    if (tid == 0) phase_join(s, j);
    __syncthreads();
    phase_hist(s, j, tid);
    __syncthreads();
    if (tid == 0 || tid == 32) phase_tree(s, tid ? 1 : 0);
    __syncthreads();
    if (tid == 0) phase_header(s);
    __syncthreads();
    phase_seg_bits(s, j, tid);
    __syncthreads();
    if (tid == 0) phase_scan(s, j);
    __syncthreads();
    phase_emit(s, j, tid);
    // CRC-32: thread t takes bytes [255 t, 255 t + 255) of the member laid against the END of a
    // 65,280-byte frame; the thread that holds byte 0 starts from 0xFFFFFFFF
    {
        const uint32_t shift = BLOCK - j.n;
        uint32_t reg = 0;
        for (uint32_t u = tid * SEG; u < (tid + 1) * SEG; u++) {
            if (u < shift) continue;
            const uint32_t i = u - shift;
            if (i == 0) reg = 0xFFFFFFFFu;
            reg = __ldg(a.table + ((reg ^ s.in[i]) & 0xFFu)) ^ (reg >> 8);
        }
        s.crc[tid] = reg;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t stride = 1u << k;
        if ((tid & (2 * stride - 1)) == 0) s.crc[tid] = gzd::gf_mul(a.op[k], s.crc[tid]) ^ s.crc[tid + stride];
        __syncthreads();
    }
    if (tid == 0) a.size[blockIdx.x] = write_frame(j.out, data_bytes(s, j), s.crc[0] ^ 0xFFFFFFFFu, j.n);
}

// members end to end: dst + off[k] <- slot k (off = exclusive prefix of the sizes, off[n] = total)
__global__ void __launch_bounds__(256) bgzf_pack(const Member *mem, const uint8_t *work, const uint32_t *off, uint8_t *dst)
{
    const uint32_t k = blockIdx.x;
    const uint32_t len = off[k + 1] - off[k];
    const uint8_t *src = work + mem[k].slot;
    uint8_t *d = dst + off[k];
    for (uint32_t i = threadIdx.x; i < len; i += 256) d[i] = src[i];
}

struct Copy {
    const uint8_t *src;
    uint8_t *dst;
    unsigned long long len;
};

__global__ void __launch_bounds__(256) bgzf_copy(const Copy *c)
{
    const Copy x = c[blockIdx.x];
    for (unsigned long long i = threadIdx.x; i < x.len; i += 256) x.dst[i] = x.src[i];
}

#endif  // __CUDACC__

}  // namespace bz
}  // namespace tdg
