"""Barcode splitter: one FASTQ file in, one trimmed FASTQ file per barcode out.

Drop-in for the reference's ``barcodeSplitter`` (/root/reference/tagdigger_fun.py:1286-1368):
same signature, same asserts, same messages, byte-identical output files.

The file is streamed through the GPU in blocks of raw bytes (``tdg_split_block``,
csrc/tdg_split.cuh): line ends, strip(), the barcode lookup (:1333), findAdapterSeq
(:1337-1339), the slices of sequence and quality, and the assembly of every barcode's output
bytes in input order all happen on the device; the host feeds bytes (parallel pread / parallel
inflate, csrc/tdg_feed.h), appends the returned pieces to the output files and prints the
reference's progress lines.  A block in which some sequence or quality line holds a non-ASCII
character is handled record by record on the host instead -- str.upper() and character
indices are Python's there -- with the two decisions still taken on the GPU (``tdg_split_batch``).

With ``bgzf=True`` every output file is BGZF (what bgzip writes) instead of plain text: the bytes of
both paths go to the device encoder (``tdg_split_bgzf``, csrc/tdg_bgzf.cuh), which cuts each file's
stream into 65,280-byte members whatever the blocks were, and decompressed each file equals the plain
one byte for byte.

``count_trimmed_file`` runs the same block loop and the same device front, but counts instead of
writing: every barcode's trimmed reads go through find_tags_fastq's matcher with a blank barcode
(``tdg_split_count_block``), as counting the output files would -- without the files.
"""

import csv
import ctypes
import hashlib
import io
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import _native, hostio, matchset, trimming
from .counting import _gzip_exception, get_engine

BLOCK_READS = 200000          # reads decided per GPU call on the host path
BLOCK_BYTES = 64 << 20        # bytes streamed through the device per call


def _byte_to_char_index(text, raw, index):
    """Slice index in characters for an index the device computed in bytes
    (differs only for sequence lines with non-ASCII characters)."""
    if index < 0 or index == 999 or len(raw) == len(text):
        return index
    return len(raw[:index].decode("utf-8", errors="ignore"))


class _Progress:
    """The reference's progress lines (:1353-1356), from per-record flags."""

    def __init__(self, name):
        self.name = name
        self.counts = [0, 0, 0]        # reads, with barcode and cut site, clipped on 3' end

    def one(self, has_bar, clipped):
        c = self.counts
        c[0] += 1
        c[1] += has_bar
        c[2] += clipped
        if c[0] % 1000000 == 0:
            print(self.name)
        if c[0] % 50000 == 0:
            print("Reads: {0} With barcode and cut site: {1} Clipped on 3' end: {2}".format(*c))

    def many(self, flags):
        """flags: uint8 per record, 1 = barcode and cut site, 2 = clipped."""
        c = self.counts
        n = len(flags)
        first = (c[0] // 50000 + 1) * 50000 - c[0]          # records up to the next multiple of 50,000
        if first <= n:
            bar = np.cumsum(flags & 1, dtype=np.int64)
            clip = np.cumsum((flags >> 1) & 1, dtype=np.int64)
            for k in range(first, n + 1, 50000):
                reads = c[0] + k
                if reads % 1000000 == 0:
                    print(self.name)
                print("Reads: {0} With barcode and cut site: {1} Clipped on 3' end: {2}".format(
                    reads, c[1] + int(bar[k - 1]), c[2] + int(clip[k - 1])))
            c[1] += int(bar[-1])
            c[2] += int(clip[-1])
        else:
            c[1] += int(np.count_nonzero(flags & 1))
            c[2] += int(np.count_nonzero(flags & 2))
        c[0] += n


def _decided_blocks(eng, text, barlen, cutlen):
    """Complete records of ``text`` (universal newlines), decided in blocks of BLOCK_READS on the
    GPU: the path for text the device does not slice itself.  Yields lists of (comment1, sequence,
    comment2, quality, barcode index or -1, slice2 in characters or None for no 3' trim)."""
    def decide(block):
        raws = [rec[1].encode("utf-8") for rec in block]
        bars, cuts = eng.split_batch(raws, barlen, cutlen)
        return [rec + (b, None if cut == 999 else _byte_to_char_index(rec[1], raw, cut))
                for rec, raw, b, cut in zip(block, raws, bars.tolist(), cuts.tolist())]

    block = []
    comment1 = sequence = comment2 = ""
    for lineindex, line in enumerate(io.StringIO(text, newline=None)):
        phase = lineindex % 4
        if phase == 0:
            comment1 = line.strip()
        elif phase == 1:
            sequence = line.strip().upper()
        elif phase == 2:
            comment2 = line.strip()
        else:
            block.append((comment1, sequence, comment2, line.strip()))
            if len(block) >= BLOCK_READS:
                yield decide(block)
                block = []
    if block:
        yield decide(block)


def _host_records(eng, text, barcodes, barlen, cutlen, outcons, progress):
    """Complete records of ``text``, decided on the GPU and written by Python."""
    for block in _decided_blocks(eng, text, barlen, cutlen):
        for comment1, sequence, comment2, quality, b, cut in block:
            clipped = 0
            if b > -1:
                slice1 = barlen[b]
                if cut is None:
                    slice2 = len(sequence)
                else:
                    slice2 = cut
                    clipped = 1
                head = comment1 + barcodes[b] + "\n"
                rec = head + sequence[slice1:slice2] + "\n" + ("+\n" if comment2 == "+" else head) + quality[slice1:slice2] + "\n"
                outcons[b].write(rec.encode("utf-8"))
            progress.one(1 if b > -1 else 0, clipped)


def _check_args(cutsite, barcodes, adapter):
    """barcodeSplitter's asserts (:1288-1293)."""
    assert set(cutsite) <= hostio.BASES, "Only ACGT cut sites allowed."
    assert all([set(bc) <= hostio.BASES for bc in barcodes]), "Found non-ACGT barcodes."
    assert len(adapter) == 2
    assert all([set(a[0]) <= set("ACGT^") for a in adapter])
    assert set(adapter[0][1]) <= hostio.BASES
    assert set(adapter[1][1]) <= set("[barcode]ACGT")


def _split_patterns(barcodes, cutsite):
    barcut = hostio.combine_barcode_and_cutsite(barcodes, cutsite)
    return matchset.effective_set(barcut, len(barcut))               # raises like build_sequence_tree


def _load_split(eng, patterns, barcodes, cutsite, adapter):
    """The splitter's tables on the device: barcode+cutsite lookup, trim tables (printing the
    reference's overlap messages), barcode strings."""
    tables = trimming.trim_tables(adapter, barcodes)
    eng.begin_file(patterns.patterns, patterns.index, [len(p) for p in patterns.patterns], any_base=patterns.any_base)
    eng.set_trim(tables[0], tables[1], tables[2], tables[3], tables[4])
    eng.split_begin(barcodes, len(cutsite))


def _open_input(inputFile):
    open(inputFile, "rb").close()                                    # the reference's OSError for a missing file
    try:
        return _native.Feed(inputFile, inputFile[-2:].lower() == "gz")
    except _native.TdgError as e:
        raise _gzip_exception(e.message) if e.code == _native.TDG_ERR_GZIP else OSError(e.message)


def _feed_error(e):
    """The exception the reference's reading raises for a TdgError of the block loop."""
    if e.code == _native.TDG_ERR_GZIP:
        return _gzip_exception(e.message)
    if e.code == _native.TDG_ERR_IO:
        return OSError(e.message)
    return e


def _block_loop(eng, feed, maxreads, device_block, host_block):
    """The splitter's loop over one input: blocks of up to BLOCK_BYTES from ``feed`` in pinned memory,
    the unconsumed tail carried to the front of the next block, the buffer doubled for a record longer
    than it.  ``device_block(buf, fill, eof, left)`` runs one block on the device and returns (records,
    consumed bytes, needs_host); ``host_block(text)`` takes the records of a block the device left to
    the host."""
    left = _native.limit_from_maxreads(maxreads)
    cap = 2 * BLOCK_BYTES
    buf = eng.host_alloc(cap)
    try:
        fill, eof = 0, False
        while left > 0:
            if not eof and fill < cap:
                got = feed.read_into(buf + fill, min(BLOCK_BYTES, cap - fill))
                eof = got == 0
                fill += got
            nrec, used, needs_host = device_block(buf, fill, eof, left)
            if nrec == 0:
                if eof:
                    break                                    # what is left is not a whole record
                if fill == cap:                              # a record longer than the buffer: make room
                    bigger = eng.host_alloc(2 * cap)
                    ctypes.memmove(bigger, buf, fill)
                    eng.host_free(buf)
                    buf, cap = bigger, 2 * cap
                continue
            if needs_host:
                host_block(ctypes.string_at(buf, used).decode("utf-8"))
            left -= nrec
            fill -= used
            if fill:
                ctypes.memmove(buf, buf + used, fill)
    finally:
        eng.host_free(buf)


def barcodeSplitter(inputFile, barcodes, outputFiles, cutsite="TGCAG", adapter=hostio.adapters["PstI-MspI-Hall"],
                    maxreads=500000000, device=None, bgzf=False):
    _check_args(cutsite, barcodes, adapter)
    if bgzf:
        # the counters (counting.py, the reference's find_tags_fastq) take a file for gzip by the last
        # two characters of its name: a BGZF file under another name would be read as text
        plain = [name for name in outputFiles if name[-2:].lower() != "gz"]
        if plain:
            raise ValueError("BGZF output needs file names ending in 'gz': %s" % ", ".join(plain))

    print("Building indices for rapid searching...")
    barlen = [len(bc) for bc in barcodes]
    patterns = _split_patterns(barcodes, cutsite)
    eng = get_engine(device)
    _load_split(eng, patterns, barcodes, cutsite, adapter)
    cutlen = len(cutsite)
    if bgzf:
        eng.split_bgzf(True)
    print("Done with indexing setup.")
    print(inputFile)

    feed = _open_input(inputFile)
    outcons = [open(name, mode="wb") for name in outputFiles]
    progress = _Progress(inputFile)
    pool = ThreadPoolExecutor(max_workers=8)

    def write(pieces):
        list(pool.map(lambda t: t[0].write(t[1]), [(o, p) for o, p in zip(outcons, pieces) if len(p)]))

    def device_block(buf, fill, eof, left):
        nrec, used, needs_host, pieces, flags = eng.split_block(buf, fill, eof, left)
        if nrec and not needs_host:
            write(pieces)
            progress.many(flags)
        return nrec, used, needs_host

    def host_block(text):
        if bgzf:
            parts = [io.BytesIO() for _ in outcons]
            _host_records(eng, text, barcodes, barlen, cutlen, parts, progress)
            write(eng.bgzf_append([p.getvalue() for p in parts]))
        else:
            _host_records(eng, text, barcodes, barlen, cutlen, outcons, progress)

    try:
        _block_loop(eng, feed, maxreads, device_block, host_block)
        if bgzf:
            write(eng.bgzf_finish())
    except _native.TdgError as e:
        raise _feed_error(e)
    finally:
        pool.shutdown()
        feed.close()
        for o in outcons:
            o.close()
    return None


def count_trimmed_file(eng, inputFile, barcodes, rows, plan, cutsite="TGCAG", adapter=hostio.adapters["PstI-MspI-Hall"],
                       maxreads=500000000):
    """barcodeSplitter(inputFile, barcodes, files, cutsite, adapter, maxreads), then
    find_tags_fastq(files[b], [''], tags, stage-2 cut site) added into matrix row ``rows[b]`` for every
    barcode b -- without the files: the splitter's device front decides every record, and the
    counter's matcher runs on the slice the file would hold (``tdg_split_count_block``).  ``plan`` is
    ``matchset.plan([''], tags, stage-2 cut site)``; the engine must hold its tags (``set_tags``) and
    the matrix.  Blocks with non-ASCII sequence or quality lines are cut by Python, as
    barcodeSplitter writes them, and counted on the GPU (``tdg_split_count_batch``).

    Returns [reads, reads with barcode and cut site, reads clipped on the 3' end, reads with tag]."""
    _check_args(cutsite, barcodes, adapter)
    barlen = [len(bc) for bc in barcodes]
    cutlen = len(cutsite)
    _load_split(eng, _split_patterns(barcodes, cutsite), barcodes, cutsite, adapter)
    eng.split_count_begin(plan.bar.patterns, plan.bar_tag_off, rows, any_base=plan.bar.any_base)
    feed = _open_input(inputFile)
    tot = [0, 0, 0, 0]

    def device_block(buf, fill, eof, left):
        nrec, used, needs_host, t = eng.split_count_block(buf, fill, eof, left)
        if nrec and not needs_host:
            for k in range(4):
                tot[k] += t[k]
        return nrec, used, needs_host

    def host_block(text):
        for block in _decided_blocks(eng, text, barlen, cutlen):
            seqs, bars = [], []
            for _c1, sequence, _c2, _q, b, cut in block:
                tot[0] += 1
                if b > -1:
                    tot[1] += 1
                    tot[2] += cut is not None
                    # the line find_tags_fastq reads back from barcode b's file: line.strip().upper()
                    seqs.append(sequence[barlen[b]:len(sequence) if cut is None else cut].strip().upper())
                    bars.append(b)
            if seqs:
                tot[3] += int(np.count_nonzero(eng.split_count_batch(seqs, bars) >= 0))

    try:
        _block_loop(eng, feed, maxreads, device_block, host_block)
    except _native.TdgError as e:
        raise _feed_error(e)
    finally:
        feed.close()
    return tot


def writeMD5sums(filelist, outfile):
    """CSV of file names and MD5 checksums (tagdigger_fun.py:1370-1386)."""
    width = max([len(f) for f in filelist])
    with open(outfile, mode="w", newline="") as con:
        w = csv.writer(con)
        w.writerow(["File name", "MD5 sum"])
        for f in filelist:
            md5 = hashlib.md5()
            with open(f, "rb") as fq:
                for chunk in iter(lambda: fq.read(50 * 1048576), b""):
                    md5.update(chunk)
            w.writerow([f, md5.hexdigest()])
            print("{:>{width}} {}".format(f, md5.hexdigest(), width=width))
    return None
