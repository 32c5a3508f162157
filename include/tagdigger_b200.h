/*
 * tagdigger_b200 -- C ABI of the B200-native TagDigger read-counting path.
 *
 * The reference (lvclark/tagdigger, pure Python) has no FFI layer.  The seam this
 * library plugs into is the plain call
 *     tagdigger_fun.find_tags_fastq(fqfile, barcodes, tags, cutsite, maxreads)
 * (tagdigger_fun.py:192-277) made once per FASTQ file from
 * tagdigger_script.py:123-126 and tagdigger_interactive.py:110-112, whose
 * results are merged by combineReadCounts (tagdigger_fun.py:1061-1098).
 * Each entry point below names the reference lines it replaces.  Signatures use
 * plain pointers and sizes only; the Python binding is ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every function returns TDG_OK (0) or a negative TDG_ERR_* code and never
 *     throws or aborts; tdg_last_error() returns the message for the last failure;
 *   - the caller owns every host buffer it passes and every output buffer;
 *     the context owns all device and pinned memory it allocates;
 *   - a context is bound to one CUDA device and is not thread-safe: one
 *     submitting host thread per context (= per GPU);
 *   - sequences are ASCII A/C/G/T (upper case), concatenated, with an offsets
 *     array of n+1 entries (CSR style);
 *   - there is no CPU implementation behind this ABI: without a CUDA device
 *     tdg_create fails.
 */
#ifndef TAGDIGGER_B200_H
#define TAGDIGGER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* The splitter's BGZF entry points (tdg_split_bgzf, tdg_bgzf_append, tdg_bgzf_finish) were added
 * to version 2 without changing any existing signature or behaviour: every version-2 caller keeps
 * working, and the version stays 2 because the test suite pins the ABI at 2.  A library built
 * before them fails at symbol lookup when the binding loads it, not silently. */
#define TDG_ABI_VERSION 2

#define TDG_OK            0
#define TDG_ERR_CUDA     -1   /* a CUDA runtime call failed (message has the CUDA error string) */
#define TDG_ERR_ARG      -2   /* invalid argument */
#define TDG_ERR_IO       -3   /* file could not be opened / read */
#define TDG_ERR_STATE    -4   /* call made out of order (e.g. submit before begin_file) */
#define TDG_ERR_NOMEM    -5
#define TDG_ERR_GZIP     -6   /* not a gzip stream / corrupt stream */
#define TDG_ERR_UTF8     -7   /* tdg_count_file: the file is not valid UTF-8 (the reference reads in text mode) */

/* flags for tdg_set_tags / tdg_begin_file */
#define TDG_ANY_BASE      1u  /* the pattern set is the single empty pattern: matches
                                 iff the next character is A/C/G/T, consuming nothing
                                 (tagdigger_fun.py:109-110) */

/* what preceded byte 0 of a chunk (tdg_count_device) */
#define TDG_PREV_NONE     0   /* start of file: byte 0 starts a line */
#define TDG_PREV_LF       1   /* the previous byte ended a line: byte 0 starts a line */
#define TDG_PREV_CR       2   /* the previous byte was '\r': it ended a line unless byte 0 is '\n' */
#define TDG_PREV_OTHER    3   /* byte 0 continues a line that started earlier */

#define TDG_LINE_CHAINED  UINT64_MAX  /* take line_base/prev_kind from the previous chunk on this context */

/* ALLOCATION SLACK the device-resident entry points need from their caller -- not the kernel's
 * geometry.  A device image of n bytes passed to tdg_count_device / tdg_count_lines_device must
 * be 16-byte aligned and sit in an allocation of at least
 *     round_up(n, TDG_TILE_BYTES) + TDG_HALO_BYTES
 * bytes (the bulk copies of the last tile read up to the next 16-byte boundary past n; the
 * rest is never touched).  The kernel's own tile and halo (csrc/tdg_kernel.cuh: 7,680 and up
 * to 256 bytes today) are smaller and may change from release to release without touching this
 * contract; the library checks at compile time that they stay below these two numbers. */
#define TDG_TILE_BYTES    16384u
#define TDG_HALO_BYTES    512u

typedef struct tdg_ctx tdg_ctx;

int         tdg_abi_version(void);

/* Create a context on CUDA device `device`.  `chunk_bytes` is the largest piece
 * tdg_submit / tdg_count_file move at once (0 = default 64 MiB); no single text
 * line may be longer than that. */
int         tdg_create(tdg_ctx **out, int device, size_t chunk_bytes);
void        tdg_destroy(tdg_ctx *ctx);
/* Message for the most recent failure on `ctx` (or of tdg_create if ctx is NULL). */
const char *tdg_last_error(const tdg_ctx *ctx);

/* The effective tag set: what build_sequence_tree(tags, len(tags))
 * (tagdigger_fun.py:98-113, :233) leaves reachable after its conflict rules,
 * i.e. a prefix-free list.  col[i] is the column of the count matrix that tag i
 * feeds (the index the reference's trie would return).  The host computes the
 * effective set (tagdigger_b200/matchset.py); this call packs it 2 bits per
 * base and builds the device hash table.  A set that is not prefix-free is
 * refused (TDG_ERR_ARG). */
int         tdg_set_tags(tdg_ctx *ctx, const char *bases, const uint64_t *off,
                         const int32_t *col, uint32_t ntags, uint32_t flags);

/* The int32 count matrix [rows x cols] (mycounts, tagdigger_fun.py:237; rows are
 * GLOBAL sample rows so the per-file matrices of tagdigger_script.py:123-126
 * never materialise).  tdg_set_matrix allocates and zeroes it; tdg_bind_matrix
 * uses caller-owned device memory instead (e.g. a torch tensor that is later
 * all-reduced with NCCL) and does not touch its contents. */
int         tdg_set_matrix(tdg_ctx *ctx, uint32_t rows, uint32_t cols);
int         tdg_bind_matrix(tdg_ctx *ctx, void *dev_int32, uint32_t rows, uint32_t cols);
int         tdg_zero_matrix(tdg_ctx *ctx);

/* Barcode+cutsite patterns of the file about to be streamed: the effective
 * (reachable, prefix-free) part of barcut (tagdigger_fun.py:213-219), each with
 * the matrix row it counts into and the offset at which tag comparison starts
 * (barcutlen, :209 and :231).  Patterns are at most 32 bases.  Resets the line
 * counter and the per-file totals. */
int         tdg_begin_file(tdg_ctx *ctx, const char *bases, const uint32_t *off,
                           const int32_t *row, const uint32_t *tag_off,
                           uint32_t npat, uint32_t flags);

/* Start the same file (same barcode table) again: resets the line counter and the
 * per-file totals only. */
int         tdg_reset_file(tdg_ctx *ctx);

/* Stream raw (uncompressed) FASTQ bytes from HOST memory: H2D copies and the
 * counting kernel, pipelined over `chunk_bytes` pieces.  Successive calls for one
 * file must pass the file's bytes in order; a trailing partial line is carried
 * over to the next call inside the context.  Returns once `bytes` may be reused
 * (kernels may still be running).  `reads_limit` is the number of reads of this
 * file to process in total (the reference's maxreads, :272-273, converted by the
 * host to max(1, ceil(maxreads))).  Replaces the loop at :250-274. */
int         tdg_submit(tdg_ctx *ctx, const void *bytes, size_t n, uint64_t reads_limit);
/* End of the current file: processes the carried partial last line. */
int         tdg_end_file(tdg_ctx *ctx, uint64_t reads_limit);

/* One chunk that is already resident in DEVICE memory (16-byte aligned).  The
 * allocation behind `dev_bytes` must extend to at least
 *   round_up(n, TDG_TILE_BYTES) + TDG_HALO_BYTES
 * bytes (contents past n are ignored).  `line_base` is the index the next line
 * START receives and `prev_kind` (TDG_PREV_*) says what preceded byte 0; pass
 * TDG_LINE_CHAINED to continue from the previous chunk on this context.  A line
 * that is cut by the end of the chunk is matched against the bytes present only,
 * so callers cut chunks at line ends (tdg_submit does).  Asynchronous. */
int         tdg_count_device(tdg_ctx *ctx, const void *dev_bytes, size_t n,
                             uint64_t line_base, int prev_kind, uint64_t reads_limit);

/* Count only the line ends of a device-resident chunk (no matching): fills
 * state[0] = line_base for the chunk that follows, state[1] = its prev_kind.
 * Used to shard one file across GPUs.  Synchronises. */
int         tdg_count_lines_device(tdg_ctx *ctx, const void *dev_bytes, size_t n,
                                   uint64_t line_base, int prev_kind, uint64_t state[2]);

/* Whole file (replaces open / gzip.open + the loop, tagdigger_fun.py:240-277): `gz` non-zero = the
 * file is gzip -- the reference decides that by the last two characters of the name, :240; the
 * binding passes that decision.  Plain files are read by host threads into pinned buffers and
 * copied to the device piece by piece.  Ordinary gzip files of 8 MiB and more are inflated ON THE
 * DEVICE (csrc/tdg_gzdev.cuh: the compressed bytes cross PCIe, thousands of lanes enter the one
 * deflate stream speculatively at block starts -- or, for BGZF files, inflate one member each --,
 * the text is born in HBM and counted there); small files, reads behind a `reads_limit`, and the
 * rest of any stream that holds something
 * the device feed does not judge (stored data it cannot enter, a damaged or truncated stream, a
 * header with unusual flags) are inflated by host threads (csrc/tdg_pgz.h, csrc/tdg_feed.h), which
 * resume at exactly the bit the device feed reached -- so every error is raised by one code path:
 * TDG_ERR_GZIP with zlib's words, which the binding maps to EOFError / zlib.error / BadGzipFile
 * like gzip.open.  TDG_GZDEV=0 in the environment keeps all inflating on the host.
 * totals: reads, reads with barcode+cutsite, reads with tag, text lines. */
int         tdg_count_file(tdg_ctx *ctx, const char *path, int gz,
                           uint64_t reads_limit, uint64_t totals[4]);

/* tdg_count_file with a look at what comes next: `next_path` (may be null) names the file the caller
 * will count after this one; its reading thread is started now, into a second set of pinned
 * buffers, so that a key of many small files (config 3; the counting stage of config 5) never
 * waits for a read.  Files the device gzip feed takes are not read ahead.  Nothing is lost when the
 * next call names another file: the reader is dropped. */
int         tdg_count_file2(tdg_ctx *ctx, const char *path, int gz, uint64_t reads_limit, uint64_t totals[4],
                            const char *next_path, int next_gz);

/* How the last tdg_count_file fed its file: info[0] rounds of the device gzip feed, [1] chunks (or BGZF
 * members) accepted, [2] 0 = the whole file went through the device, 1 = the host feeder took over
 * somewhere, -1 = host feeder only. */
int         tdg_last_file_info(tdg_ctx *ctx, int64_t info[3]);

/* Frees the working buffers of the device-side gzip feed (tokens, symbols, windows, text: about ten
 * times the compressed bytes of a round, at most ~12 GB) and the staging buffer of tdg_trim_batch,
 * tdg_split_batch and tdg_match_batch; they are kept between calls otherwise. */
int         tdg_release_scratch(tdg_ctx *ctx);

/* The gzip feed of tdg_count_file by itself (tests, profiling): inflates `path` into the host
 * buffer dst[0..cap) -- rounds on the device, the rest, if any, through the host feeder -- and
 * reports the number of bytes in *n.  info: [0] device rounds, [1] chunks run, [2] chunks accepted,
 * [3] 0 = everything on the device, 1 = the host's parallel reader resumed, 2 = zlib resumed,
 * -1 = not a file the device feed takes; ms (may be null): milliseconds of upload, scan, decode,
 * windows + resolve, CRC fold, copy-out.  Errors as tdg_count_file. */
int         tdg_gz_inflate_host(tdg_ctx *ctx, const char *path, void *dst, size_t cap, uint64_t *n,
                                int64_t info[4], double ms[6]);

/* Wait for all submitted work. */
int         tdg_sync(tdg_ctx *ctx);
/* Running totals since the last tdg_begin_file (synchronises): reads, reads with
 * barcode+cutsite, reads with tag, text lines started. */
int         tdg_file_totals(tdg_ctx *ctx, uint64_t totals[4]);
/* Synchronise and copy the matrix to host (`out` may be NULL to skip). */
int         tdg_read_matrix(tdg_ctx *ctx, int32_t *out);

/* Overflow guard.  Cells are int32 on the device while the reference counts with unbounded
 * Python integers (tagdigger_fun.py:237,266): *out receives the smallest cell of the matrix --
 * counts only grow, so a negative value means that some cell passed INT32_MAX since the matrix
 * was zeroed (callers raise OverflowError; see tagdigger_b200/counting.py).  Synchronous. */
int         tdg_matrix_min(tdg_ctx *ctx, int32_t *out);

/* Multi-GPU: one context per GPU (one process or thread each).  The only exchange of the path
 * is the sum of the per-GPU matrices -- the cross-file sum of combineReadCounts
 * (tagdigger_fun.py:1088-1095) taken across GPUs -- done as ONE ncclAllReduce(int32, sum), in
 * place, on the context's stream, i.e. in stream order behind the last count kernel and ahead
 * of the next tdg_zero_matrix / tdg_read_matrix.  NCCL is bound at run time (libnccl.so.2).
 *   tdg_comm_unique_id   rank 0 makes the 128-byte id and hands it to the other ranks
 *                        (any channel: MPI, a file, torch.distributed ...)
 *   tdg_comm_init        every rank joins (collective: blocks until all ranks have called)
 *   tdg_allreduce_matrix asynchronous; a no-op on a context without communicator
 *   tdg_finish           all-reduce, then the totals of this rank and the matrix on the host
 *                        (the SURVEY's tdg_finish: sync, all-reduce, D2H) */
int         tdg_comm_unique_id(void *out128);
int         tdg_comm_init(tdg_ctx *ctx, const void *id128, int nranks, int rank);
int         tdg_allreduce_matrix(tdg_ctx *ctx);
int         tdg_finish(tdg_ctx *ctx, int32_t *out, uint64_t totals[4]);

/* Device pointer of the matrix and the CUDA stream the kernels run on, so the
 * caller can all-reduce the matrix in place (NCCL) right behind the last kernel:
 * the multi-GPU replacement for the sum in combineReadCounts (:1081-1097). */
void       *tdg_matrix_device_ptr(tdg_ctx *ctx);
void       *tdg_stream(tdg_ctx *ctx);
/* Make the context's stream wait for work already queued on `other_stream`, or
 * `other_stream` wait for the context's stream (handles are cudaStream_t passed
 * as void*; NULL is the legacy default stream), for in-stream collectives. */
int         tdg_stream_wait(tdg_ctx *ctx, void *other_stream);
int         tdg_other_stream_wait(tdg_ctx *ctx, void *other_stream);

/* Pinned host memory for callers that want tdg_submit to DMA straight from
 * their buffer. */
void       *tdg_host_alloc(tdg_ctx *ctx, size_t n);
void        tdg_host_free(tdg_ctx *ctx, void *p);
/* Plain device memory (for tdg_count_device callers without another allocator). */
void       *tdg_device_alloc(tdg_ctx *ctx, size_t n);
void        tdg_device_free(tdg_ctx *ctx, void *p);
int         tdg_memcpy_h2d(tdg_ctx *ctx, void *dev, const void *host, size_t n);
int         tdg_memcpy_d2h(tdg_ctx *ctx, void *host, const void *dev, size_t n);

/* Number of kernels this context has launched (bench.py's gpu_launches). */
uint64_t    tdg_launch_count(const tdg_ctx *ctx);
/* Device time in milliseconds of the counting kernels launched between
 * tdg_timing_begin and tdg_timing_end (CUDA events on the context's stream,
 * one pair per kernel launch; at most 4096 launches), of the BGZF writer's
 * kernels (one pair per deflate-scan-pack sequence) and of every
 * tdg_split_count_block (one pair around its upload and kernels).  tdg_timing_end
 * synchronises; *nlaunch receives the number of kernels timed. */
int         tdg_timing_begin(tdg_ctx *ctx);
int         tdg_timing_end(tdg_ctx *ctx, double *kernel_ms, uint32_t *nlaunch);

/* Trim decision of the barcode splitter (findAdapterSeq, tagdigger_fun.py:1251-1283,
 * with the tables of build_adapter_tree, :1208-1249).  The host passes the two full
 * restriction sites (common cutter, rare cutter), the common-cutter string a0 (site
 * remnant + adapter), one rare-cutter string per barcode (a1, CSR offsets) and, per
 * barcode, the REACHABLE adapter prefixes of the reference's reversed trie as
 * (which string, length, slice index) triples -- tagdigger_b200/trimming.py derives
 * them, including the reference's overlap fallback (:1237-1248). */
int         tdg_set_trim(tdg_ctx *ctx, const char *site0, const char *site1, const char *a0,
                         uint32_t nbar, const char *a1, const uint32_t *a1_off,
                         const uint32_t *cand_off, const uint16_t *cand_len,
                         const int16_t *cand_idx, const uint8_t *cand_which);
/* slice2[i] = findAdapterSeq(seq_i, tables[bar[i]], site0, site1, start[i]) for n
 * sequence lines given as HOST buffers (already stripped; case is folded on the
 * device): position after the first full site at or after start[i] (the earlier of
 * the two, the rare cutter on a tie), else the negative slice index of the adapter
 * prefix the read ends with, else 999.  One warp per read; synchronous. */
int         tdg_trim_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, const int32_t *bar,
                           const uint32_t *start, uint32_t n, int32_t *slice2);

/* The two decisions barcodeSplitter takes per read (tagdigger_fun.py:1333-1343), for n
 * sequence lines given as HOST buffers (stripped; case is folded on the device):
 * bar_out[i] = sequence_index_lookup(seq_i, barcuttree) -- the barcode table is the one
 * loaded by tdg_begin_file with rows = barcode indices -- and, where that is >= 0,
 * slice2[i] = findAdapterSeq(seq_i, adaptertrees[bar], site0, site1, bar_len[bar] + cutlen)
 * (tables from tdg_set_trim); 999 elsewhere.  One warp per read; synchronous. */
int         tdg_split_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, uint32_t n,
                            const uint32_t *bar_len, uint32_t nbar, uint32_t cutlen,
                            int32_t *bar_out, int32_t *slice2);

/* Streaming barcode splitter: the loop of barcodeSplitter (tagdigger_fun.py:1327-1363) for one
 * block of raw, uncompressed FASTQ bytes, entirely on the device -- universal-newline line
 * ends, strip() of the four lines, barcode lookup (:1333), findAdapterSeq (:1337-1339), the
 * Python slices sequence[slice1:slice2] / quality[slice1:slice2] (:1346,:1351), and the bytes
 * each barcode's output file gains, in input order.
 * tdg_split_begin: the barcode strings (appended to the first line, :1345) and the cut-site
 * length; needs tdg_begin_file (barcode+cutsite table, rows = barcode indices) and
 * tdg_set_trim.
 * tdg_split_block: `bytes` (host, n <= 1 GiB) must start at a record boundary; final_block
 * != 0 when the file ends with it (a last line without terminator is then a line).  At most
 * max_records records are taken.  *n_records = complete records handled, *consumed = bytes
 * they span (the caller carries the rest over to the front of its next block).
 * *needs_host = 1: some record has a non-ASCII byte in its sequence or quality line
 * (str.upper() and character indices are Python's then); nothing was produced and the
 * caller handles bytes[0 .. consumed) itself.  Otherwise out[out_off[b] .. out_off[b+1]) are
 * the bytes to append to barcode b's file and flags[r] = 1 (barcode and cut site found)
 * | 2 (clipped on the 3' end) for every record; the three pointers are pinned host memory
 * owned by the context, valid until the next call.  With BGZF output on (tdg_split_bgzf), out /
 * out_off carry the completed BGZF members of every barcode's file instead of plain bytes. */
int         tdg_split_begin(tdg_ctx *ctx, const char *barcodes, const uint32_t *bar_off, uint32_t nbar,
                            uint32_t cutlen);
int         tdg_split_block(tdg_ctx *ctx, const uint8_t *bytes, size_t n, int final_block,
                            uint64_t max_records, uint64_t *n_records, uint64_t *consumed,
                            int *needs_host, const uint8_t **out, const uint64_t **out_off,
                            const uint8_t **flags);

/* Counting the streaming splitter's output instead of writing it: barcodeSplitter(f, barcodes,
 * files, cutsite=S1, adapter=A) followed by find_tags_fastq(files[b], [''], tags, cutsite) for every
 * barcode b, with barcode b's counts added to matrix row row_of_barcode[b] -- in one pass, without
 * the files.  The stage-2 line of a record is t = sequence[slice1:slice2].strip() (upper case).
 * tdg_split_count_begin: after tdg_set_tags, a matrix and tdg_split_begin (tdg_split_begin drops
 * it again); loads the stage-2 barcode+cutsite table (blank barcode: the patterns, tag offsets and
 * flags tdg_begin_file takes, without rows) and row_of_barcode[nbar], every row inside the matrix.
 * The stage-1 table of tdg_begin_file stays as it is.
 * tdg_split_count_block: as tdg_split_block for *n_records, *consumed and *needs_host; instead of
 * output bytes, every record's tag hit is added to the matrix and totals[] receives the block's
 * reads, reads with barcode and cut site, reads clipped on the 3' end and reads with a tag.  With
 * *needs_host = 1 the matrix is untouched and totals[] are 0: the caller decides the records with
 * tdg_split_batch, cuts t itself and counts it with tdg_split_count_batch.
 * tdg_split_count_batch: n stage-2 lines t_i given as HOST buffers (stripped, upper case) with
 * their stage-1 barcodes bar[i] (0 <= bar[i] < nbar); adds the hits to the matrix and returns
 * col_out[i] = the tag column or -1.  Synchronous. */
int         tdg_split_count_begin(tdg_ctx *ctx, const char *bases, const uint32_t *off, const uint32_t *tag_off,
                                  uint32_t npat, uint32_t flags, const int32_t *row_of_barcode);
int         tdg_split_count_block(tdg_ctx *ctx, const uint8_t *bytes, size_t n, int final_block,
                                  uint64_t max_records, uint64_t *n_records, uint64_t *consumed,
                                  int *needs_host, uint64_t totals[4]);
int         tdg_split_count_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, const int32_t *bar,
                                  uint32_t n, int32_t *col_out);

/* BGZF output files for the streaming splitter (the reference writes plain text only).  Every
 * barcode's file is the series of gzip members bgzip writes: member k holds bytes
 * [k * 65280, (k+1) * 65280) of the file's uncompressed stream (the last one may be short), with the
 * `BC` extra field (FLG = 4, XLEN = 6, BSIZE = member size - 1), CRC32 and ISIZE; a member is at
 * most 65,536 bytes (a dynamic-Huffman block, or stored blocks when those are not larger).  The cuts
 * depend on the stream alone: every barcode's pending tail (< 65,280 bytes) is kept in the context
 * between calls, and tdg_split_block and tdg_bgzf_append append to the same streams, in call order.
 * tdg_split_bgzf: after tdg_split_begin; on != 0 switches BGZF output on and empties the tails
 * (on = 0 switches it off; tdg_split_begin does too).
 * tdg_bgzf_append: bytes[off[b] .. off[b+1]) (host memory, nbar + 1 offsets, at most 1 GiB in all)
 * are appended to barcode b's stream -- the records the caller wrote itself after needs_host.
 * tdg_bgzf_finish: the tails become the last members and every file ends with the 28-byte BGZF
 * end-of-file member (a barcode without reads gets that member alone); the tails are empty after.
 * Both return, like tdg_split_block, out[out_off[b] .. out_off[b+1]) = the bytes to append to
 * barcode b's file, in pinned host memory owned by the context and valid until the next call. */
int         tdg_split_bgzf(tdg_ctx *ctx, int on);
int         tdg_bgzf_append(tdg_ctx *ctx, const uint8_t *bytes, const uint64_t *off,
                            const uint8_t **out, const uint64_t **out_off);
int         tdg_bgzf_finish(tdg_ctx *ctx, const uint8_t **out, const uint64_t **out_off);

/* The host feed by itself (what tdg_count_file reads through): the uncompressed bytes of a
 * plain, gzip or BGZF file -- gzip.open(f, 'rt') / open(f, 'r') of tagdigger_fun.py:240-243
 * and :1316-1319 -- with parallel pread / parallel inflate on host threads (TDG_IO_THREADS).
 * No context; errors via tdg_last_error(NULL).  tdg_feed_read returns the bytes written to
 * dst (0 = end of file) or a negative TDG_ERR_* code. */
typedef struct tdg_feed tdg_feed;
int         tdg_feed_open(tdg_feed **out, const char *path, int gz);
long long   tdg_feed_read(tdg_feed *feed, void *dst, size_t cap);
void        tdg_feed_close(tdg_feed *feed);

/* Per-read results of the matcher for n sequence lines given as HOST buffers (stripped;
 * case is folded on the device): row_out[i] = the barcode row (sequence_index_lookup on
 * barcuttree, tagdigger_fun.py:257) or -1, col_out[i] = the tag column (:260-261) or -1.
 * For callers that must see individual reads: find_tags_fastq(tassel_tagcount=True) adds
 * the count= weight of each read's header line (:251-253, :264-265) on the host.
 * Uses the tables of tdg_set_tags / tdg_begin_file; synchronous. */
int         tdg_match_batch(tdg_ctx *ctx, const char *seqs, const uint64_t *off, uint32_t n,
                            int32_t *row_out, int32_t *col_out);

/* CSV output with host threads, for count matrices held as int32 arrays (writeCounts,
 * tagdigger_fun.py:1100-1111, and writeDiploidGeno, :1144-1180; byte-identical to Python's
 * csv.writer).  `header` is the finished header line including "\r\n"; row r starts with
 * labels[label_off[r] .. label_off[r+1]) (the CSV-escaped sample name), followed by
 * ",cell" for every column and "\r\n".  Genotype cells: '0' if only the marker's allele-0
 * column is > 0, '1' if both, '2' if only allele 1, empty otherwise.  No context needed;
 * on failure the message is returned by tdg_last_error(NULL). */
int         tdg_write_counts_csv(const char *path, const int32_t *matrix, uint32_t rows, uint32_t cols,
                                 const char *header, size_t header_len, const char *labels,
                                 const uint64_t *label_off, int threads);
int         tdg_write_geno_csv(const char *path, const int32_t *matrix, uint32_t rows, uint32_t cols,
                               const uint32_t *col0, const uint32_t *col1, uint32_t nmarkers,
                               const char *header, size_t header_len, const char *labels,
                               const uint64_t *label_off, int threads);

#ifdef __cplusplus
}
#endif
#endif /* TAGDIGGER_B200_H */
