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
``count_trimmed_resident`` counts the same way on text that is already in device memory
(``tdg_split_count_device``): one rank's share of a file sharded across GPUs.

``split_files`` splits every file of a key, and under torchrun cuts one large library file into one
share per GPU: each rank sizes its share's output on the device (``tdg_split_device`` with sizes_only),
the ranks exchange the sizes, and each writes its bytes at their offsets in the same output files.
"""

import contextlib
import csv
import ctypes
import hashlib
import io
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import _native, counting, hostio, matchset, trimming
from .counting import _reference_error, get_engine

BLOCK_READS = 200000          # reads decided per GPU call on the host path
BLOCK_BYTES = 64 << 20        # bytes streamed through the device per call


def _byte_to_char_index(text, raw, index):
    """Slice index in characters for an index the device computed in bytes
    (differs only for sequence lines with non-ASCII characters)."""
    if index < 0 or index == 999 or len(raw) == len(text):
        return index
    return len(raw[:index].decode("utf-8", errors="ignore"))


class _Progress:
    """The reference's progress lines (:1353-1356), from per-record flags.  ``counts`` start at ``start``
    (the totals of the records before these: a later rank's share of a sharded file) and every line goes
    to ``out`` (print by default)."""

    def __init__(self, name, start=(0, 0, 0), out=print):
        self.name = name
        self.counts = list(start)      # reads, with barcode and cut site, clipped on 3' end
        self.out = out

    def one(self, has_bar, clipped):
        c = self.counts
        c[0] += 1
        c[1] += has_bar
        c[2] += clipped
        if c[0] % 1000000 == 0:
            self.out(self.name)
        if c[0] % 50000 == 0:
            self.out("Reads: {0} With barcode and cut site: {1} Clipped on 3' end: {2}".format(*c))

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
                    self.out(self.name)
                self.out("Reads: {0} With barcode and cut site: {1} Clipped on 3' end: {2}".format(
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
        raise _reference_error(e, opening=True)


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


def _set_up_split(inputFile, barcodes, outputFiles, cutsite, adapter, device, bgzf):
    """barcodeSplitter's checks, set-up and first lines (:1288-1326): returns the engine, its split tables
    loaded."""
    _check_args(cutsite, barcodes, adapter)
    if bgzf:
        # the counters (counting.py, the reference's find_tags_fastq) take a file for gzip by the last
        # two characters of its name: a BGZF file under another name would be read as text
        plain = [name for name in outputFiles if name[-2:].lower() != "gz"]
        if plain:
            raise ValueError("BGZF output needs file names ending in 'gz': %s" % ", ".join(plain))

    print("Building indices for rapid searching...")
    patterns = _split_patterns(barcodes, cutsite)
    eng = get_engine(device)
    _load_split(eng, patterns, barcodes, cutsite, adapter)
    if bgzf:
        eng.split_bgzf(True)
    print("Done with indexing setup.")
    print(inputFile)
    return eng


def barcodeSplitter(inputFile, barcodes, outputFiles, cutsite="TGCAG", adapter=hostio.adapters["PstI-MspI-Hall"],
                    maxreads=500000000, device=None, bgzf=False):
    eng = _set_up_split(inputFile, barcodes, outputFiles, cutsite, adapter, device, bgzf)
    barlen = [len(bc) for bc in barcodes]
    cutlen = len(cutsite)
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
        raise _reference_error(e)
    finally:
        pool.shutdown()
        feed.close()
        for o in outcons:
            o.close()
    return None


def split_files(bckeys, cutsite, adapter, maxreads=500000000, bgzf=False, device=None, rank=0, world=1, gather=None):
    """Every input file of a splitter key (``readBarcodeKeyfile(..., forSplitter=True)``: {input file: [barcodes,
    output files]}) through barcodeSplitter: the loop of barcode_splitter_script, in sorted order at
    ``world == 1``.

    With ``world > 1`` (one process per GPU) and fewer files than ranks, the files :func:`counting.shard_files`
    picks (plain files of at least SHARD_MIN_BYTES per rank, clean BGZF member chains) are split by all ranks
    together (:func:`_split_sharded`, which needs ``gather(list) -> list of every rank's list``,
    :func:`counting.dist_gather`), and go first; the others are dealt whole (:func:`counting.assign_files`),
    each printed by the rank that splits it.  The output files are byte for byte those of one rank, and rank 0
    prints a sharded file's lines as one rank would.  With ``bgzf`` every file is dealt whole: member cuts of
    an output file depend on everything before them."""
    files = sorted(bckeys.keys())
    split = {} if bgzf else counting.shard_files(files, world)
    todo = list(split) + counting.assign_files([f for f in files if f not in split], rank, world)
    for f in todo:
        barcodes, outputs = bckeys[f][0], bckeys[f][1]
        if f in split:
            _split_sharded(f, barcodes, outputs, cutsite, adapter, maxreads, device, rank, world, gather, split[f])
        else:
            barcodeSplitter(f, barcodes, outputs, cutsite=cutsite, adapter=adapter, maxreads=maxreads, device=device,
                            bgzf=bgzf)


class _SplitShards(counting._RecordShards):
    """Placement of a sharded file's ranges for the splitter: on record boundaries, ``maxreads`` records in all."""

    def __init__(self, maxreads):
        self.maxreads = maxreads


def shard_offsets(per_rank, rank):
    """The element-wise sum of the rows of the ranks before ``rank``: with rows of every barcode's output
    bytes, where rank ``rank``'s bytes start in each barcode's file; with rows of totals, the totals the
    progress lines of its records start from."""
    out = [0] * (len(per_rank[0]) if per_rank else 0)
    for row in per_rank[:rank]:
        out = [a + int(b) for a, b in zip(out, row)]
    return out


def _split_sharded(inputFile, barcodes, outputFiles, cutsite, adapter, maxreads, device, rank, world, gather, index):
    """barcodeSplitter(inputFile, barcodes, outputFiles, cutsite, adapter, maxreads) by all ranks at once, each
    on its own share of the file (``index``: its BGZF member index, None for a plain file):

    1. set-up as barcodeSplitter's, its lines kept back; the steps of :func:`counting._place_share` (load,
       line count, first ``gather``, record-aligned placement); if some rank cannot take part, rank 0
       splits the file whole with barcodeSplitter and the other ranks skip it;
    2. pass 1 sizes every barcode's share of the rank's records (``split_device`` with sizes_only);
    3. rank 0 creates or truncates the output files; a second ``gather`` of [failed, sizes, totals] gives
       every rank its offset in each output file and the totals before its first record;
    4. pass 2 writes its records at those offsets (``os.pwrite``) and composes its progress lines;
    5. a third ``gather`` of [failed, lines]: rank 0 prints barcodeSplitter's first lines and then every
       rank's lines in rank order.
    A rank that fails in 2 or 4 raises its own exception after the next gather, the others a RuntimeError
    naming it; no rank writes after a failed pass 1."""
    preamble = io.StringIO()
    try:
        with contextlib.redirect_stdout(preamble):
            eng = _set_up_split(inputFile, barcodes, outputFiles, cutsite, adapter, device, False)
    except BaseException:
        if rank == 0:
            print(preamble.getvalue(), end="")
        raise
    placed = counting._place_share(eng, _SplitShards(maxreads), inputFile, rank, world, gather, index)
    if placed is None:
        if rank == 0:
            barcodeSplitter(inputFile, barcodes, outputFiles, cutsite=cutsite, adapter=adapter, maxreads=maxreads,
                            device=device)
        return
    dev, n, (start, tail, _first, max_records) = placed
    share = (eng, dev + start, n - start + len(tail), max_records, inputFile, barcodes, [len(bc) for bc in barcodes],
             len(cutsite))
    nbar = len(barcodes)
    lines = []
    try:
        sizes, tot, err = [0] * nbar, [0, 0, 0], None
        try:
            if tail:
                eng.memcpy_h2d(dev + n, np.frombuffer(tail, dtype=np.uint8).ctypes.data, len(tail))
            sizes, tot = _size_share(*share)
            if rank == 0:
                for name in outputFiles:
                    open(name, "wb").close()
        except Exception as e:                  # every rank still takes part in the gather
            err = _reference_error(e) if isinstance(e, _native.TdgError) else e
        every = counting._gather_checked(gather, inputFile, err, sizes + tot, "splitting")
        offsets = shard_offsets([x[:nbar] for x in every], rank)
        err = None
        try:
            ends = _write_share(*share, outputFiles, offsets, shard_offsets([x[nbar:] for x in every], rank), lines.append)
            if ends != [a + b for a, b in zip(offsets, sizes)]:
                raise RuntimeError("%s: the bytes written differ from the bytes sized" % inputFile)
        except Exception as e:
            err = _reference_error(e) if isinstance(e, _native.TdgError) else e
        every = counting._gather_checked(gather, inputFile, err, lines, "splitting")
    finally:
        eng.device_free(dev)
        if rank == 0:
            print(preamble.getvalue(), end="")
    if rank == 0:
        for rank_lines in every:
            for line in rank_lines:
                print(line)


def _size_share(eng, dev, n, max_records, name, barcodes, barlen, cutlen):
    """Pass 1 of _split_sharded over the ``n`` bytes of text at ``dev``: (bytes every barcode's file gains,
    [reads, with barcode and cut site, clipped on the 3' end])."""
    sizes = np.zeros(len(barcodes), dtype=np.int64)
    tot = [0, 0, 0]

    def device_call(p, size, final, left):
        nrec, used, needs_host, offs, _flags, t = eng.split_device(p, size, final, left, sizes_only=True)
        if nrec and not needs_host:
            sizes[:] += np.diff(offs.astype(np.int64))
            for k in range(3):
                tot[k] += t[k]
        return nrec, used, needs_host

    def host_block(text):
        sinks = [_Sized() for _ in barcodes]
        progress = _Progress(name, out=lambda line: None)
        _host_records(eng, text, barcodes, barlen, cutlen, sinks, progress)
        for b, sink in enumerate(sinks):
            sizes[b] += sink.n
        for k in range(3):
            tot[k] += progress.counts[k]

    _resident_loop(eng, dev, n, max_records, device_call, host_block, "split_files")
    return [int(x) for x in sizes], tot


def _write_share(eng, dev, n, max_records, name, barcodes, barlen, cutlen, outputFiles, offsets, start, out):
    """Pass 2 of _split_sharded: the records of the text at ``dev`` written into the output files from
    ``offsets`` on, their progress lines (counted from ``start``) sent to ``out``.  Returns the offsets
    every file was written up to."""
    progress = _Progress(name, start, out)
    files = []
    pool = ThreadPoolExecutor(max_workers=8)
    try:
        for path, off in zip(outputFiles, offsets):
            files.append(_FileAt(os.open(path, os.O_WRONLY), off))

        def device_call(p, size, final, left):
            nrec, used, needs_host, pieces, flags, _t = eng.split_device(p, size, final, left)
            if nrec and not needs_host:
                list(pool.map(lambda t: t[0].put(t[1]), [(f, x) for f, x in zip(files, pieces) if len(x)]))
                progress.many(flags)
            return nrec, used, needs_host

        def host_block(text):
            _host_records(eng, text, barcodes, barlen, cutlen, files, progress)
            for f in files:
                f.flush()

        _resident_loop(eng, dev, n, max_records, device_call, host_block, "split_files")
    finally:
        pool.shutdown()
        for f in files:
            os.close(f.fd)
    return [f.off for f in files]


class _Sized:
    """A sink that counts the bytes written to it (pass 1's host path)."""

    def __init__(self):
        self.n = 0

    def write(self, data):
        self.n += len(data)


class _FileAt:
    """An output file written from offset ``off`` on: ``write`` collects the host path's records until
    ``flush``, ``put`` writes a piece at once; both with os.pwrite, so ranks write one file side by side."""

    def __init__(self, fd, off):
        self.fd, self.off, self.pending = fd, off, []

    def write(self, data):
        self.pending.append(data)

    def flush(self):
        if self.pending:
            self.put(b"".join(self.pending))
            self.pending = []

    def put(self, data):
        view = memoryview(data).cast("B")
        while len(view):
            k = os.pwrite(self.fd, view, self.off)
            if k <= 0:
                raise OSError("short write to output file")
            self.off += k
            view = view[k:]


def _trimmed_counter(eng, barcodes, rows, plan, cutsite, adapter):
    """The set-up of a one-pass count (split tables, stage-2 table) and the two block handlers that
    count_trimmed_file and count_trimmed_resident share.  Returns (tot, device_result, host_block):
    ``tot`` = [reads, with barcode and cut site, clipped on the 3' end, with tag] so far;
    ``device_result(r)`` adds the totals of a split_count_block / split_count_device result r and
    returns (records, consumed, needs_host); ``host_block(text)`` cuts and counts the records of a
    block the device left to the host."""
    _check_args(cutsite, barcodes, adapter)
    barlen = [len(bc) for bc in barcodes]
    cutlen = len(cutsite)
    _load_split(eng, _split_patterns(barcodes, cutsite), barcodes, cutsite, adapter)
    eng.split_count_begin(plan.bar.patterns, plan.bar_tag_off, rows, any_base=plan.bar.any_base)
    tot = [0, 0, 0, 0]

    def device_result(r):
        nrec, used, needs_host, t = r
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

    return tot, device_result, host_block


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
    tot, device_result, host_block = _trimmed_counter(eng, barcodes, rows, plan, cutsite, adapter)
    feed = _open_input(inputFile)

    def device_block(buf, fill, eof, left):
        return device_result(eng.split_count_block(buf, fill, eof, left))

    try:
        _block_loop(eng, feed, maxreads, device_block, host_block)
    except _native.TdgError as e:
        raise _reference_error(e)
    finally:
        feed.close()
    return tot


RESIDENT_CALL_BYTES = 1 << 30     # the split kernels' 32-bit offsets: at most 1 GiB per tdg_split_count_device call


def count_trimmed_resident(eng, dev, n, barcodes, rows, plan, cutsite, adapter, max_records):
    """count_trimmed_file on text already in device memory: ``n`` bytes at ``dev`` that begin at a record
    start and end at a record boundary or at the end of the file, of which at most ``max_records``
    records are taken.  The text is walked in calls of at most RESIDENT_CALL_BYTES
    (``tdg_split_count_device``), each starting where the previous one stopped; the last call is final.
    A call that needs the host copies its bytes back and goes through count_trimmed_file's host path.
    Returns the same four totals."""
    tot, device_result, host_block = _trimmed_counter(eng, barcodes, rows, plan, cutsite, adapter)
    _resident_loop(eng, dev, n, max_records, lambda p, size, final, left: device_result(
        eng.split_count_device(p, size, final, left)), host_block, "count_trimmed_resident")
    return tot


def _resident_loop(eng, dev, n, max_records, device_call, host_block, what):
    """The walk over resident text that count_trimmed_resident and split_files' passes share: calls of at
    most RESIDENT_CALL_BYTES, each starting where the previous one stopped, the last one final.
    ``device_call(ptr, size, final, left)`` runs one call and returns (records, consumed, needs_host); a call
    that needs the host copies its bytes back and hands their text to ``host_block``."""
    pos = done = 0
    while pos < n and done < max_records:
        size = min(RESIDENT_CALL_BYTES, n - pos)
        final = pos + size == n
        nrec, used, needs_host = device_call(dev + pos, size, final, max_records - done)
        if nrec == 0:
            if final:
                break                                        # what is left is not a whole record
            raise _native.TdgError(_native.TDG_ERR_ARG, "%s: a record longer than %d bytes" % (what, RESIDENT_CALL_BYTES))
        if needs_host:
            raw = np.empty(used, dtype=np.uint8)
            eng.memcpy_d2h(raw.ctypes.data, dev + pos, used)
            host_block(raw.tobytes().decode("utf-8"))
        done += nrec
        pos += used


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
