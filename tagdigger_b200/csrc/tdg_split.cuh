// Streaming barcode splitter on the device (sm_100a): one block of raw FASTQ bytes in, the
// bytes of every barcode's output file for that block out.
//
// Replaces the loop of barcodeSplitter, /root/reference/tagdigger_fun.py:1327-1363:
//   for line in fqcon:                                   -> line ends of the block (universal
//       lineindex % 4 == 0..3: strip(), upper()             newlines), numbered by a prefix sum
//       barindex = sequence_index_lookup(...)            -> match_barcode (tdg_match.h)
//       slice2 = findAdapterSeq(...)                     -> trim_decide (tdg_trim.cuh)
//       outcons[barindex].write(...) x 4                 -> record sizes, a per-barcode prefix sum
//                                                           in input order, byte copies
// Kernels, in launch order:
//   lineend_count   line ends per 4 KiB tile
//   tile_scan       exclusive prefix over the tile counts (one CTA)
//   lineend_scatter ends[i] = byte position of the terminator of line i
//   split_records   one warp per record: strip the four lines, barcode, trim decision, Python
//                   slice arithmetic, output size; records whose sequence or quality line holds
//                   a non-ASCII byte raise the block's `complex` flag (str.upper() and character
//                   indices are the host's business then)
//   bar_tile_sums   output bytes per (tile of 256 records, barcode)
//   bar_tile_scan   per barcode: exclusive prefix over the tiles, totals, barcode bases
//   split_write     per tile: in-order offsets of its records inside their barcode's stream,
//                   then the bytes
// Sizing a block without writing it (tdg_split_device with sizes_only): the same front up to
// split_records, then
//   split_tally     output bytes per barcode and the three flag counts of the block
//
// Counting the trimmed reads without writing them (tdg_split_count_block): the same front up to
// split_records, then
//   split_count     one thread per record: find_tags_fastq's matcher (match_line, tdg_match.h) on
//                   the stripped slice sequence[slice1:slice2] -- what the counter would read back
//                   from the barcode's output file -- with the stage-2 table (blank barcode), the
//                   hit added to the matrix row of the record's barcode; totals of the block
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "tdg_match.h"
#include "tdg_trim.cuh"

namespace tdg {

constexpr uint32_t SPLIT_TILE_BYTES = 4096;     // 256 threads x 16 bytes
constexpr uint32_t SPLIT_REC_TILE = 256;        // records per CTA in the output kernels
constexpr uint32_t SPLIT_FLAG_BAR = 1, SPLIT_FLAG_CLIP = 2;

struct SplitRec {             // one FASTQ record of the block, after the decisions
    uint32_t c1, c1_len;      // stripped first line
    uint32_t seq, seq_len;    // slice of the sequence line that is written
    uint32_t qual, qual_len;  // slice of the quality line that is written
    int32_t bar;              // barcode index or -1
    uint32_t plus_bare;       // 1: third line is exactly "+"
};

struct SplitBlock {
    const uint8_t *bytes;
    uint32_t n;               // bytes in the block
    uint32_t final_block;     // 1: the file ends with this block
    uint32_t n_tiles;
    uint32_t *tile_count;     // [n_tiles + 1] counts, then exclusive prefix; [n_tiles] = total
    uint32_t *ends;           // [lines] terminator position of every line (n for an unterminated last line)
    uint32_t ends_cap;
};

struct SplitWork {
    SplitBlock b;
    uint32_t n_rec;
    SplitRec *rec;            // [n_rec]
    uint8_t *flags;           // [n_rec] SPLIT_FLAG_*
    uint32_t *complex_flag;   // set when a record needs the host
    SplitArgs s;              // tables: s.t (trim), s.bar, s.bar_len, s.cutlen
    const uint8_t *barcodes;  // concatenated barcode strings
    const uint32_t *bar_off;  // [nbar + 1]
    uint32_t nbar;
    uint32_t n_rtiles;
    uint32_t *tile_sums;      // [n_rtiles][nbar] bytes, then exclusive prefix per barcode
    unsigned long long *bar_base;   // [nbar + 1] start of every barcode's stream in out
    uint8_t *out;
};

// The counter's side of split_count / split_count_batch
struct SplitCountArgs {
    const BarTable *bar;      // stage-2 barcode+cutsite table: find_tags_fastq(F_i, [''], tags, cutsite)
    TagTable tags;
    const int32_t *row_of;    // [nbar] matrix row of every stage-1 barcode
    int32_t *matrix;
    uint32_t cols;
};

#if defined(__CUDACC__)

// 16 bytes -> 16-bit mask of line ends: '\n', or '\r' that is not followed by '\n'
// (`next` = the byte after these 16; 0x100 = there is none and the file goes on: undecided)
__device__ __forceinline__ uint32_t lineend_mask16(uint4 q, uint32_t next)
{
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const uint32_t c = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
        const uint32_t nx = i < 15 ? (w[(i + 1) >> 2] >> (8 * ((i + 1) & 3))) & 0xFFu : next;
        const bool end = c == '\n' || (c == '\r' && nx != '\n' && nx != 0x100u);
        m |= (uint32_t)end << i;
    }
    return m;
}

// mask of thread `tid`'s 16 bytes (bytes at and past n do not exist)
__device__ __forceinline__ uint32_t split_thread_mask(const SplitBlock &b, uint32_t unit)
{
    const uint32_t p = unit * 16u;
    if (p >= b.n) return 0;
    const uint4 q = *(const uint4 *)(b.bytes + p);                 // the allocation is padded to 16
    uint32_t next;
    if (p + 16 < b.n) next = b.bytes[p + 16];
    else next = b.final_block ? 0u : 0x100u;
    uint32_t m = lineend_mask16(q, next);
    const uint32_t valid = b.n - p;
    if (valid < 16) {
        m &= (1u << valid) - 1u;
        // the last existing byte: a '\r' there is followed by nothing
        const uint32_t c = b.bytes[b.n - 1];
        if (c == '\r') {
            if (b.final_block) m |= 1u << (valid - 1);
            else m &= ~(1u << (valid - 1));
        }
    }
    return m;
}

__global__ void __launch_bounds__(256) lineend_count(const SplitBlock b)
{
    __shared__ uint32_t wsum[8];
    const uint32_t unit = blockIdx.x * 256u + threadIdx.x;
    uint32_t c = __popc(split_thread_mask(b, unit));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if ((threadIdx.x & 31u) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int i = 0; i < 8; i++) t += wsum[i];
        b.tile_count[blockIdx.x] = t;
    }
}

// in-place exclusive prefix over v[0..n), total in v[n]; one CTA of 1024 threads
__global__ void __launch_bounds__(1024) tile_scan(uint32_t *v, uint32_t n)
{
    __shared__ uint32_t part[1024];
    const uint32_t tid = threadIdx.x;
    const uint32_t per = (n + 1023u) / 1024u;
    const uint32_t lo = tid * per, hi = lo + per < n ? lo + per : n;
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += v[i];
    part[tid] = sum;
    __syncthreads();
    for (uint32_t d = 1; d < 1024; d <<= 1) {
        const uint32_t x = tid >= d ? part[tid - d] : 0;
        __syncthreads();
        part[tid] += x;
        __syncthreads();
    }
    uint32_t run = part[tid] - sum;
    for (uint32_t i = lo; i < hi; i++) {
        const uint32_t c = v[i];
        v[i] = run;
        run += c;
    }
    if (tid == 1023) v[n] = part[1023];
}

__global__ void __launch_bounds__(256) lineend_scatter(const SplitBlock b)
{
    __shared__ uint32_t wsum[8];
    const uint32_t unit = blockIdx.x * 256u + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t m = split_thread_mask(b, unit);
    const uint32_t c = __popc(m);
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= (uint32_t)d) incl += o;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    uint32_t base = b.tile_count[blockIdx.x];
    for (uint32_t w = 0; w < warp; w++) base += wsum[w];
    uint32_t idx = base + incl - c;
    while (m) {
        const uint32_t bit = __ffs(m) - 1u;
        m &= m - 1u;
        if (idx < b.ends_cap) b.ends[idx] = unit * 16u + bit;
        idx++;
    }
}

__device__ __forceinline__ bool split_is_space(uint32_t c)      // str.strip() for ASCII
{
    return is_lead_space(c) || c == '\n' || c == '\r';
}

// [lo, hi) -> the same range without leading and trailing whitespace (str.strip(), including
// the UTF-8 encoded Unicode spaces)
__device__ __forceinline__ void split_strip(const uint8_t *s, uint32_t &lo, uint32_t &hi)
{
    for (;;) {
        if (lo >= hi) return;
        const uint32_t c = s[lo];
        if (split_is_space(c)) { lo++; continue; }
        if (c >= 0xC2 && c <= 0xE3 && lo + 1 < hi) {
            const uint32_t u = utf8_space(c, s[lo + 1], lo + 2 < hi ? s[lo + 2] : 0u);
            if (u && lo + u <= hi) { lo += u; continue; }
        }
        break;
    }
    for (;;) {
        if (lo >= hi) return;
        const uint32_t c = s[hi - 1];
        if (split_is_space(c)) { hi--; continue; }
        if (c >= 0x80) {
            if (hi - lo >= 2 && utf8_space(s[hi - 2], c, 0u) == 2u) { hi -= 2; continue; }
            if (hi - lo >= 3 && utf8_space(s[hi - 3], s[hi - 2], c) == 3u) { hi -= 3; continue; }
        }
        break;
    }
}

// Python's s[a:b] for a >= 0 and any b on a string of length n: (start, length)
__device__ __forceinline__ void py_slice(uint32_t n, uint32_t a, int32_t b, uint32_t &start, uint32_t &len)
{
    const uint32_t lo = a < n ? a : n;
    uint32_t hi;
    if (b < 0) hi = (uint32_t)(-b) < n ? n - (uint32_t)(-b) : 0u;
    else hi = (uint32_t)b < n ? (uint32_t)b : n;
    start = lo;
    len = hi > lo ? hi - lo : 0u;
}

__global__ void __launch_bounds__(256) split_records(const SplitWork w)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t r = blockIdx.x * 8u + (threadIdx.x >> 5);
    if (r >= w.n_rec) return;
    const uint8_t *s = w.b.bytes;
    uint32_t lo[4], hi[4];
#pragma unroll
    for (uint32_t k = 0; k < 4; k++) {
        const uint32_t li = 4u * r + k;
        lo[k] = li ? w.b.ends[li - 1] + 1u : 0u;
        hi[k] = w.b.ends[li];
        split_strip(s, lo[k], hi[k]);
    }
    // sequence and quality lines must be ASCII for the device to slice them by bytes
    bool high = false;
    for (uint32_t p = lo[1] + lane; p < hi[1]; p += 32) high |= s[p] >= 0x80;
    for (uint32_t p = lo[3] + lane; p < hi[3]; p += 32) high |= s[p] >= 0x80;
    if (__any_sync(0xFFFFFFFFu, high)) {
        if (lane == 0) {
            *w.complex_flag = 1u;
            SplitRec none;
            none.c1 = none.c1_len = none.seq = none.seq_len = none.qual = none.qual_len = none.plus_bare = 0;
            none.bar = -1;
            w.rec[r] = none;
            w.flags[r] = 0;
        }
        return;
    }
    const uint32_t n = hi[1] - lo[1];
    int32_t b = -1;
    {
        GlobalBytes f;
        f.p = s + lo[1];
        f.limit = n;
        const BarEntry *bent = (const BarEntry *)((const uint8_t *)w.s.bar + sizeof(BarTable));
        b = match_barcode(f, w.s.bar, bent);
    }
    int32_t cut = TRIM_NONE;
    if (b >= 0) cut = trim_decide(w.s.t, s + lo[1], n, w.s.bar_len[b] + w.s.cutlen, b, lane);
    if (lane == 0) {
        SplitRec rec;
        rec.c1 = lo[0];
        rec.c1_len = hi[0] - lo[0];
        rec.bar = b;
        rec.plus_bare = (hi[2] - lo[2] == 1u && s[lo[2]] == '+') ? 1u : 0u;
        rec.seq = rec.seq_len = rec.qual = rec.qual_len = 0;
        uint8_t fl = 0;
        if (b >= 0) {
            fl = SPLIT_FLAG_BAR;
            const uint32_t slice1 = w.s.bar_len[b];
            int32_t slice2 = cut;
            if (cut == TRIM_NONE) slice2 = (int32_t)n;          // :1340-1341
            else fl |= SPLIT_FLAG_CLIP;
            uint32_t st, ln;
            py_slice(n, slice1, slice2, st, ln);
            rec.seq = lo[1] + st;
            rec.seq_len = ln;
            py_slice(hi[3] - lo[3], slice1, slice2, st, ln);
            rec.qual = lo[3] + st;
            rec.qual_len = ln;
        }
        w.rec[r] = rec;
        w.flags[r] = fl;
    }
}

// bytes record `rec` adds to its barcode's file (:1345-1351)
__device__ __forceinline__ uint32_t split_out_len(const SplitRec &rec, const uint32_t *bar_off)
{
    if (rec.bar < 0) return 0;
    const uint32_t head = rec.c1_len + (bar_off[rec.bar + 1] - bar_off[rec.bar]) + 1u;
    return head + rec.seq_len + 1u + (rec.plus_bare ? 2u : head) + rec.qual_len + 1u;
}

__global__ void __launch_bounds__(SPLIT_REC_TILE) bar_tile_sums(const SplitWork w)
{
    extern __shared__ uint32_t sums[];          // [nbar]
    for (uint32_t i = threadIdx.x; i < w.nbar; i += SPLIT_REC_TILE) sums[i] = 0;
    __syncthreads();
    const uint32_t r = blockIdx.x * SPLIT_REC_TILE + threadIdx.x;
    if (r < w.n_rec) {
        const SplitRec rec = w.rec[r];
        if (rec.bar >= 0) atomicAdd(&sums[rec.bar], split_out_len(rec, w.bar_off));
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < w.nbar; i += SPLIT_REC_TILE) w.tile_sums[(size_t)blockIdx.x * w.nbar + i] = sums[i];
}

// one thread per barcode walks the tiles; then thread 0 lays the barcodes' streams end to end
__global__ void __launch_bounds__(256) bar_tile_scan(const SplitWork w, unsigned long long *bar_total)
{
    const uint32_t b = blockIdx.x * 256u + threadIdx.x;
    if (b >= w.nbar) return;
    unsigned long long run = 0;
    for (uint32_t t = 0; t < w.n_rtiles; t++) {
        const uint32_t c = w.tile_sums[(size_t)t * w.nbar + b];
        // offsets inside one block fit 32 bits: a block is < 4 GiB and a record at most doubles
        w.tile_sums[(size_t)t * w.nbar + b] = (uint32_t)run;
        run += c;
    }
    bar_total[b] = run;
}

__global__ void bar_bases(const unsigned long long *bar_total, unsigned long long *bar_base, uint32_t nbar)
{
    if (blockIdx.x || threadIdx.x) return;
    unsigned long long run = 0;
    for (uint32_t b = 0; b < nbar; b++) {
        bar_base[b] = run;
        run += bar_total[b];
    }
    bar_base[nbar] = run;
}

// Sizes only (tdg_split_device with sizes_only): the bytes every barcode's file gains from the block and
// its three flag counts, without offsets or output.  Each CTA walks records grid-stride, sums output bytes
// per barcode in shared memory (32-bit, as bar_tile_scan's in-block offsets) and adds its non-zero sums to
// tally[0 .. nbar); tally[nbar + 0..2] gain reads, reads with barcode and cut site, reads clipped on the
// 3' end.  A block split_records left to the host (complex flag) is not tallied: the host sizes it.
__global__ void __launch_bounds__(SPLIT_REC_TILE) split_tally(const SplitWork w, unsigned long long *tally)
{
    if (*w.complex_flag) return;
    extern __shared__ uint32_t sums[];          // [nbar]
    __shared__ uint32_t part[3][SPLIT_REC_TILE / 32];
    for (uint32_t i = threadIdx.x; i < w.nbar; i += SPLIT_REC_TILE) sums[i] = 0;
    __syncthreads();
    uint32_t v[3] = {0, 0, 0};
    for (uint32_t r = blockIdx.x * SPLIT_REC_TILE + threadIdx.x; r < w.n_rec; r += gridDim.x * SPLIT_REC_TILE) {
        const SplitRec rec = w.rec[r];
        const uint8_t fl = w.flags[r];
        v[0] += 1;
        v[1] += fl & SPLIT_FLAG_BAR ? 1u : 0u;
        v[2] += fl & SPLIT_FLAG_CLIP ? 1u : 0u;
        if (rec.bar >= 0) atomicAdd(&sums[rec.bar], split_out_len(rec, w.bar_off));
    }
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint32_t s = __reduce_add_sync(0xFFFFFFFFu, v[k]);
        if (lane == 0) part[k][warp] = s;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < w.nbar; i += SPLIT_REC_TILE)
        if (sums[i]) atomicAdd(tally + i, (unsigned long long)sums[i]);
    if (threadIdx.x < 3) {
        unsigned long long s = 0;
        for (uint32_t i = 0; i < SPLIT_REC_TILE / 32; i++) s += part[threadIdx.x][i];
        if (s) atomicAdd(tally + w.nbar + threadIdx.x, s);
    }
}

__device__ __forceinline__ void split_copy(uint8_t *dst, const uint8_t *src, uint32_t n, uint32_t lane, bool upper)
{
    for (uint32_t i = lane; i < n; i += 32) {
        uint32_t c = src[i];
        if (upper) c = fold_upper(c);
        dst[i] = (uint8_t)c;
    }
}

__global__ void __launch_bounds__(SPLIT_REC_TILE) split_write(const SplitWork w)
{
    extern __shared__ uint32_t running[];       // [nbar] next free offset of every barcode's stream in this tile
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t tile = blockIdx.x;
    for (uint32_t i = threadIdx.x; i < w.nbar; i += SPLIT_REC_TILE) running[i] = w.tile_sums[(size_t)tile * w.nbar + i];
    const uint32_t r = tile * SPLIT_REC_TILE + threadIdx.x;
    SplitRec rec;
    rec.c1 = rec.c1_len = rec.seq = rec.seq_len = rec.qual = rec.qual_len = rec.plus_bare = 0;
    rec.bar = -1;
    if (r < w.n_rec) rec = w.rec[r];
    const uint32_t len = rec.bar >= 0 ? split_out_len(rec, w.bar_off) : 0u;
    uint32_t my_off = 0;
    __syncthreads();
    // ---- offsets in input order: the warps take turns, inside a warp lane order decides
    for (uint32_t turn = 0; turn < SPLIT_REC_TILE / 32; turn++) {
        if (warp == turn) {
            uint32_t before = 0, group = 0;
            bool first = true;
            for (uint32_t j = 0; j < 32; j++) {
                const int32_t bj = __shfl_sync(0xFFFFFFFFu, rec.bar, j);
                const uint32_t lj = __shfl_sync(0xFFFFFFFFu, len, j);
                if (bj == rec.bar) {
                    group += lj;
                    if (j < lane) { before += lj; first = false; }
                }
            }
            if (rec.bar >= 0) my_off = running[rec.bar] + before;
            __syncwarp();
            if (rec.bar >= 0 && first) running[rec.bar] += group;
        }
        __syncthreads();
    }
    // ---- bytes: a warp writes its 32 records one after the other, all lanes on one record
    const uint8_t *s = w.b.bytes;
    for (uint32_t j = 0; j < 32; j++) {
        const int32_t bj = __shfl_sync(0xFFFFFFFFu, rec.bar, j);
        const uint32_t off = __shfl_sync(0xFFFFFFFFu, my_off, j);
        const uint32_t c1 = __shfl_sync(0xFFFFFFFFu, rec.c1, j), c1_len = __shfl_sync(0xFFFFFFFFu, rec.c1_len, j);
        const uint32_t sq = __shfl_sync(0xFFFFFFFFu, rec.seq, j), sq_len = __shfl_sync(0xFFFFFFFFu, rec.seq_len, j);
        const uint32_t ql = __shfl_sync(0xFFFFFFFFu, rec.qual, j), ql_len = __shfl_sync(0xFFFFFFFFu, rec.qual_len, j);
        const uint32_t bare = __shfl_sync(0xFFFFFFFFu, rec.plus_bare, j);
        if (bj < 0) continue;
        const uint8_t *bc = w.barcodes + w.bar_off[bj];
        const uint32_t blen = w.bar_off[bj + 1] - w.bar_off[bj];
        uint8_t *dst = w.out + w.bar_base[bj] + off;
        const uint32_t head = c1_len + blen + 1u;
        split_copy(dst, s + c1, c1_len, lane, false);               // comment1 + barcode  (:1345)
        split_copy(dst + c1_len, bc, blen, lane, false);
        if (lane == 0) dst[head - 1] = '\n';
        dst += head;
        split_copy(dst, s + sq, sq_len, lane, true);                // sequence[slice1:slice2], upper case  (:1346)
        if (lane == 0) dst[sq_len] = '\n';
        dst += sq_len + 1u;
        if (bare) {                                                 // '+'  (:1347-1348)
            if (lane == 0) { dst[0] = '+'; dst[1] = '\n'; }
            dst += 2;
        } else {                                                    // or the first line again  (:1349-1350)
            split_copy(dst, s + c1, c1_len, lane, false);
            split_copy(dst + c1_len, bc, blen, lane, false);
            if (lane == 0) dst[head - 1] = '\n';
            dst += head;
        }
        split_copy(dst, s + ql, ql_len, lane, false);               // quality[slice1:slice2]  (:1351)
        if (lane == 0) dst[ql_len] = '\n';
    }
}

// The counter's rule on one stage-2 line t (stripped): its tag column, or -1.  The window ends where t
// ends, so a tag cannot reach past slice2.  Case is folded by the matcher (t.upper()).
__device__ __forceinline__ int32_t split_count_col(const SplitCountArgs &c, const uint8_t *p, uint32_t len)
{
    GlobalBytes f;
    f.p = p;
    f.limit = len;
    const BarEntry *bent = (const BarEntry *)((const uint8_t *)c.bar + sizeof(BarTable));
    const MatchResult m = match_line(f, c.bar, bent, c.tags);
    return m.row >= 0 ? m.col : -1;
}

// counts[row_of[bar]][col] += 1 for every lane that has a hit (bar >= 0, col >= 0); lanes on the same
// cell add together, once.  Every lane of the warp must call it.
__device__ __forceinline__ void split_count_add(const SplitCountArgs &c, int32_t bar, int32_t col)
{
    const bool hit = bar >= 0 && col >= 0;
    // cells < 2^32 - 1 (tdg_set_matrix): the all-ones key is no cell
    const uint32_t cell = hit ? (uint32_t)c.row_of[bar] * c.cols + (uint32_t)col : 0xFFFFFFFFu;
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cell);
    if (hit && (threadIdx.x & 31u) == (uint32_t)__ffs(peers) - 1u) atomicAdd(c.matrix + cell, (int)__popc(peers));
}

// One thread per record of the block (after split_records): the trimmed sequence slice, stripped,
// through the counter's matcher into the matrix.  totals[0..3] gain the block's reads, reads with
// barcode and cut site, reads clipped on the 3' end and reads with a tag.  A block split_records left
// to the host (complex flag) is not counted at all: the host counts its records itself.
__global__ void __launch_bounds__(256) split_count(const SplitWork w, const SplitCountArgs c, unsigned long long *totals)
{
    if (*w.complex_flag) return;
    __shared__ uint32_t part[4][8];
    const uint32_t r = blockIdx.x * 256u + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    int32_t bar = -1, col = -1;
    uint32_t clipped = 0;
    if (r < w.n_rec) {
        const SplitRec rec = w.rec[r];
        bar = rec.bar;
        if (bar >= 0) {
            clipped = (w.flags[r] & SPLIT_FLAG_CLIP) ? 1u : 0u;
            // t = s[slice1:slice2].strip(): blanks can surface inside the slice when the cut site is empty
            uint32_t lo = rec.seq, hi = rec.seq + rec.seq_len;
            split_strip(w.b.bytes, lo, hi);
            col = split_count_col(c, w.b.bytes + lo, hi - lo);
        }
    }
    split_count_add(c, bar, col);
    const uint32_t v[4] = {r < w.n_rec ? 1u : 0u, bar >= 0 ? 1u : 0u, clipped, col >= 0 ? 1u : 0u};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t s = __reduce_add_sync(0xFFFFFFFFu, v[k]);
        if (lane == 0) part[k][warp] = s;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        uint32_t s = 0;
        for (int i = 0; i < 8; i++) s += part[threadIdx.x][i];
        if (s) atomicAdd(totals + threadIdx.x, (unsigned long long)s);
    }
}

// The same count for stage-2 lines the host cut itself (blocks left to the host):
// t_i = seqs[off[i] .. off[i+1]), stripped and upper-cased by Python; bar[i] >= 0 its stage-1 barcode.
__global__ void __launch_bounds__(128) split_count_batch(const uint8_t *seqs, const unsigned long long *off, const int32_t *bar,
                                                         uint32_t n, const SplitCountArgs c, int32_t *col_out)
{
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    int32_t b = -1, col = -1;
    if (r < n) {
        b = bar[r];
        col = split_count_col(c, seqs + off[r], (uint32_t)(off[r + 1] - off[r]));
        col_out[r] = col;
    }
    split_count_add(c, b, col);
}

#endif  // __CUDACC__

}  // namespace tdg
