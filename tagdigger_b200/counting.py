"""Host side of the counting path: the drop-in for ``find_tags_fastq``.

Mirrors /root/reference/tagdigger_fun.py:192-277 (same signature, defaults,
asserts and return shape); the per-read loop runs on the GPU through
``_native.Engine`` (ctypes over include/tagdigger_b200.h).  Nothing here counts
reads on the CPU.
"""

import ctypes
import gzip
import os
import re
import zlib

import numpy as np

from . import _native
from . import matchset

_engines = {}


def get_engine(device=None):
    """The process-wide Engine of a CUDA device (created on first use).  With
    ``device=None`` the device is LOCAL_RANK (torchrun) or 0."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    eng = _engines.get(device)
    if eng is None:
        eng = _native.Engine(device=device)
        _engines[device] = eng
    return eng


def load_plan(eng, p, row_of=None, nrows=None, set_tags=True):
    """Upload a matchset.CountPlan.  ``row_of[b]`` maps the barcode index the
    reference's trie would return to a matrix row (identity by default)."""
    if set_tags:
        eng.set_tags(p.tags.patterns, p.tags.index, any_base=p.tags.any_base)
    if nrows is not None:
        eng.set_matrix(nrows, p.ntags)
    rows = p.bar.index if row_of is None else [row_of[b] for b in p.bar.index]
    eng.begin_file(p.bar.patterns, rows, p.bar_tag_off, any_base=p.bar.any_base)


def _gzip_exception(message):
    """The exception gzip.open(...).read() of the reference (tagdigger_fun.py:240-241) raises for
    the same defect: EOFError for a stream that stops early, zlib.error for invalid deflate data,
    BadGzipFile for bad headers and CRC / length mismatches."""
    if "unexpected end of file" in message:
        return EOFError("Compressed file ended before the end-of-stream marker was reached (%s)" % message)
    if "invalid" in message or "compressed data error" in message:
        return zlib.error("Error -3 while decompressing data: %s" % message)
    return gzip.BadGzipFile(message)


def _is_gz(name):
    return name[-2:].lower() == "gz"            # tagdigger_fun.py:240


def _reference_error(e, opening=False):
    """The exception the reference's open() / gzip.open(...).read() raises (tagdigger_fun.py:240-243) for
    the defect a library call reported as TdgError ``e``: gzip's for a gzip defect, OSError for an I/O
    error, UnicodeDecodeError for invalid UTF-8 (open(f, 'r') / gzip.open(f, 'rt') decode the file; of
    the library's calls only tdg_count_file checks it).  Other codes (CUDA, allocation, state) have no
    counterpart there and stay ``e`` -- except when ``opening`` a file: the feed's open fails as
    open() does, with an OSError."""
    if e.code == _native.TDG_ERR_GZIP:
        return _gzip_exception(e.message)
    if e.code == _native.TDG_ERR_IO or opening:
        return OSError(e.message)
    if e.code == _native.TDG_ERR_UTF8:
        pos = int(e.message.split()[1].rstrip(":")) if e.message.startswith("position ") else 0
        return UnicodeDecodeError("utf-8", b"\xff", 0, 1, "invalid UTF-8 at byte %d (%s)" % (pos, e.message))
    return e


def _run_file(eng, fqfile, limit, next_file=None):
    """Stream one file; map library errors to the exceptions the reference's
    open()/gzip.open() would raise.  ``next_file``: the file that will be counted next (the
    library starts reading it while this one is counted)."""
    with open(fqfile, "rb"):                    # FileNotFoundError / PermissionError / IsADirectoryError
        pass
    try:
        return eng.count_file(fqfile, _is_gz(fqfile), limit, next_path=next_file,
                              next_gz=_is_gz(next_file) if next_file else False)
    except _native.TdgError as e:
        raise _reference_error(e)


def find_tags_fastq(fqfile, barcodes, tags, cutsite="TGCAG", maxreads=5e9, tassel_tagcount=False,
                    device=None, totals=None):
    """Count reads of ``fqfile`` per (barcode, tag): the GPU replacement of
    tagdigger_fun.find_tags_fastq (tagdigger_fun.py:192-277).  Returns a
    ``len(barcodes) x len(tags)`` list of lists of int.

    ``totals`` (optional list) receives [reads, reads with barcode and cut
    site, reads with tag] -- the running totals the reference prints."""
    p = matchset.plan(barcodes, tags, cutsite)
    if tassel_tagcount:
        return _find_tags_weighted(fqfile, p, maxreads, device, totals)
    limit = _native.limit_from_maxreads(maxreads)
    if p.barnum == 0 or p.ntags == 0:
        # the reference's trie builder indexes an empty list (tagdigger_fun.py:76)
        raise IndexError("list index out of range")
    eng = get_engine(device)
    load_plan(eng, p, nrows=p.barnum)
    tot = _run_file(eng, fqfile, limit)
    counts = eng.read_matrix()
    print("Reads: {0} With barcode and cut site: {1} With tag: {2}".format(tot[0], tot[1], tot[2]))
    if totals is not None:
        totals[:] = tot[:3]
    return counts.tolist()


TASSEL_BLOCK = 200000         # reads matched per GPU call in tassel_tagcount mode


def _find_tags_weighted(fqfile, p, maxreads, device, totals):
    """find_tags_fastq with tassel_tagcount=True (tagdigger_fun.py:251-253, :264-265): every
    header line carries ``count=N`` and a matching read adds N instead of 1.  Such files list
    each distinct tag once, so they are small; the host reads the text and evaluates
    ``int(...)`` exactly as the reference does (including its ValueError for a header without
    a parsable count), the GPU matches a block of reads per call (``tdg_match_batch``) and the
    weights are added as Python integers (no overflow)."""
    if p.barnum == 0 or p.ntags == 0:
        raise IndexError("list index out of range")
    eng = get_engine(device)
    load_plan(eng, p, nrows=p.barnum)
    counts = [[0] * p.ntags for _ in range(p.barnum)]
    tot = [0, 0, 0]

    def flush(seqs, weights):
        rows, cols = eng.match_batch(seqs)
        for r, c, w in zip(rows.tolist(), cols.tolist(), weights):
            if r > -1:
                tot[1] += 1
                if c > -1:
                    tot[2] += 1
                    counts[r][c] += w

    con = gzip.open(fqfile, "rt") if _is_gz(fqfile) else open(fqfile, "r")
    try:
        seqs, weights = [], []
        weight = 0
        for lineindex, line in enumerate(con):
            phase = lineindex % 4
            if phase == 0:
                weight = int(line[line.find("count=") + 6:].strip())
            elif phase == 1:
                tot[0] += 1
                seqs.append(line.strip().upper())
                weights.append(weight)
                if len(seqs) >= TASSEL_BLOCK:
                    flush(seqs, weights)
                    seqs, weights = [], []
                if tot[0] >= maxreads:
                    break
        if seqs:
            flush(seqs, weights)
    finally:
        con.close()
    print("Reads: {0} With barcode and cut site: {1} With tag: {2}".format(*tot))
    if totals is not None:
        totals[:] = tot
    return counts


def find_tags_bytes(data, barcodes, tags, cutsite="TGCAG", maxreads=5e9, device=None, totals=None,
                    pieces=None):
    """Same as find_tags_fastq on an in-memory FASTQ image (bytes), streamed
    through tdg_submit.  ``pieces`` optionally lists split points to submit the
    image in several calls (exercises the carry-over of partial lines)."""
    p = matchset.plan(barcodes, tags, cutsite)
    limit = _native.limit_from_maxreads(maxreads)
    eng = get_engine(device)
    load_plan(eng, p, nrows=p.barnum)
    arr = np.frombuffer(data, dtype=np.uint8)
    cuts = [0] + sorted(pieces or []) + [arr.size]
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            eng.submit(arr[a:b], limit)
    eng.end_file(limit)
    tot = eng.file_totals()
    if totals is not None:
        totals[:] = tot
    return eng.read_matrix().tolist()


def global_rows(bckeys):
    """Sample names in output order and, for every file, the matrix row of each
    of its barcodes -- the row layout combineReadCounts produces
    (tagdigger_fun.py:1061-1098): files in sorted order, samples in key-file
    order, one row per distinct sample name."""
    samples, row_of, rows = [], {}, {}
    for f in sorted(bckeys.keys()):
        mine = []
        for sample in bckeys[f][1]:
            r = row_of.get(sample)
            if r is None:
                r = row_of[sample] = len(samples)
                samples.append(sample)
            mine.append(r)
        rows[f] = mine
    return samples, rows


def count_files(bckeys, tags, cutsite="TGCAG", maxreads=5e9, device=None, rank=0, world=1, reduce=None,
                totals=None, as_array=False, gather=None, adapter=None, split_cutsite=None, split_maxreads=500000000):
    """All files of a key (``readBarcodeKeyfile`` output) in one go: the batched
    form of the loop at tagdigger_script.py:123-128.  Every file counts straight
    into the GLOBAL sample rows of one device matrix, so the result equals
    ``combineReadCounts({f: find_tags_fastq(f, ...)}, bckeys)`` without per-file
    matrices; the tag table is uploaded once.

    With ``world > 1`` (one process per GPU) the files are dealt to the ranks by
    size (largest first, to the least loaded rank) and ``reduce(ptr, rows, cols,
    engine)`` must sum the per-rank matrices in place (one NCCL all-reduce, see
    :func:`nccl_reduce`); integer sums make the result independent of ``world``.  When there are
    fewer files than ranks, plain files are sharded by byte range, and BGZF files by member range,
    instead and counted first
    (:func:`_count_sharded`, which needs ``gather(list_of_ints) -> list of every rank's list``,
    :func:`dist_gather`).  Results, rank 0's output and exceptions stay those of a one-rank run.

    Returns ``[sample names, count rows]`` -- rows as lists of int like combineReadCounts, or,
    with ``as_array=True``, as one int32 ndarray (hostio.writeCounts / writeDiploidGeno format
    that with native threads; a 384 x 500,000 matrix is 768 MB as an array and several GB as
    Python integers).  Each file prints one line with its totals, on the rank that counted it (rank 0
    for a sharded file), and ``totals`` (optional dict) receives ``{file: [reads, with barcode and
    cut site, with tag]}`` for this rank's files; a sharded file's totals are summed over the ranks
    and go to every rank (to rank 0 alone when it counted the file whole).

    With ``adapter`` (the name of an adapter set, a key of ``hostio.adapters``) every file is first
    split and trimmed as ``barcodeSplitter(f, barcodes, files, cutsite=split_cutsite, adapter=...,
    maxreads=split_maxreads)`` would, and each barcode's output is then counted as
    ``find_tags_fastq(file, [''], tags, cutsite)`` into its sample's row -- in one pass per file on the
    GPU, without writing the split files (:func:`splitter.count_trimmed_file`).  ``split_cutsite``
    defaults to the cut site of the adapter set's enzyme, as barcode_splitter_script derives it.  Files
    are dealt or sharded as above.  ``totals`` then receives ``[reads, with barcode and cut site,
    clipped on the 3' end, with tag]``."""
    files = sorted(bckeys.keys())
    samples, rows = global_rows(bckeys)
    if adapter is None:
        mode = _PlainCount(bckeys, files, rows, tags, cutsite, maxreads)
    else:
        mode = _TrimmedCount(bckeys, files, rows, tags, cutsite, maxreads, adapter, split_cutsite, split_maxreads)
    eng = get_engine(device)
    eng.set_tags(mode.tags.patterns, mode.tags.index, any_base=mode.tags.any_base)
    eng.set_matrix(len(samples), len(tags))
    split = shard_files(files, world)
    todo = list(split) + assign_files([f for f in files if f not in split], rank, world)
    for i, f in enumerate(todo):
        if f in split:
            tot = _count_sharded(eng, mode, f, rank, world, gather, split[f])
            if tot is None:
                continue                          # rank 0 counted the file whole
        else:
            tot = mode.whole(eng, f, next_file=todo[i + 1] if i + 1 < len(todo) else None)
        if rank == 0 or f not in split:
            print(mode.line.format(f, *tot))
        if totals is not None:
            totals[f] = tot
    return _result(eng, samples, len(tags), world, reduce, as_array)


def _result(eng, samples, ntags, world, reduce, as_array):
    """count_files' return value: the matrix, summed over the ranks."""
    if world > 1:
        if reduce is None:
            raise ValueError("count_files with world > 1 needs a reduce callable (see nccl_reduce)")
        reduce(eng.matrix_ptr(), len(samples), ntags, eng)
    matrix = eng.read_matrix()
    return [samples, matrix if as_array else matrix.tolist()]


class _PlainCount:
    """count_files' plain mode: every file counted as find_tags_fastq counts it.  Construction runs the
    set-up checks, file by file, before anything is counted.  What the mode supplies to count_files and
    :func:`_count_sharded`: ``tags`` (the tag plan), ``line`` (the format of a file's output line),
    ``whole`` (count a whole file), ``payload`` / ``extra`` / ``place`` (what a rank adds to the
    first gather, the room it needs behind its range, and where its range lies in the file), ``own``
    (count its range) and ``ascii_only`` (a range of a BGZF file with a byte >= 0x80 is not sharded)."""
    line = "{0}: Reads: {1} With barcode and cut site: {2} With tag: {3}"
    extra = 0
    ascii_only = True         # tdg_count_device does not check UTF-8 (DESIGN §7): sharded BGZF text stays ASCII

    def __init__(self, bckeys, files, rows, tags, cutsite, maxreads):
        self.limit = _native.limit_from_maxreads(maxreads)
        self.rows = rows
        self.plans = {}
        tagplan = None
        for f in files:
            if tagplan is None:
                self.plans[f] = matchset.plan(bckeys[f][0], tags, cutsite)
                tagplan = matchset.plan_tags(tags, cutsite)       # shared by the other files of the key
            else:
                self.plans[f] = matchset.plan(bckeys[f][0], tags, cutsite, tagplan=tagplan)
            if self.plans[f].barnum == 0 or self.plans[f].ntags == 0:
                raise IndexError("list index out of range")
        self.tags = self.plans[files[0]].tags

    def whole(self, eng, f, next_file=None):
        """[reads, with barcode and cut site, with tag] of file ``f``."""
        load_plan(eng, self.plans[f], row_of=self.rows[f], set_tags=False)
        return _run_file(eng, f, self.limit, next_file)[:3]

    def payload(self, head):
        return []

    def place(self, lines, payloads, rank):
        """The range's first line index in the file: read indices, and so ``maxreads``, stay global."""
        return sum(lines[:rank])

    def own(self, eng, f, rank, dev, n, base):
        load_plan(eng, self.plans[f], row_of=self.rows[f], set_tags=False)   # a fresh line state, too
        eng.count_device(dev, n, base, _native.TDG_PREV_NONE if rank == 0 else _native.TDG_PREV_LF, self.limit)
        return eng.file_totals()[:3]


class _RecordShards:
    """How a sharded file is placed when its ranges must be cut on RECORD boundaries (the splitter's device
    front decides whole records): the members ``extra`` / ``payload`` / ``place`` / ``ascii_only`` of
    :class:`_PlainCount` for the one-pass mode and for :func:`splitter.split_files`.  ``maxreads`` is the
    split's record limit."""
    ascii_only = False        # non-ASCII records go to the host (the split entry points' needs_host)

    @property
    def extra(self):
        return HEAD_CAP           # room for the lines of the next range that complete the last record

    def payload(self, head):
        """The range's head (``head()``: :func:`range_head` for a plain file, the loaded text's for a BGZF
        file), or None when it is too long to send."""
        h = head()
        return None if h is None else list(h)

    def place(self, lines, payloads, rank):
        """The range's owned text and record budget (:func:`plan_trimmed_shards`); None to handle the file whole."""
        shards = plan_trimmed_shards(lines, [bytes(p) for p in payloads], _native.limit_from_maxreads(self.maxreads))
        return None if shards is None else shards[rank]


class _TrimmedCount(_RecordShards):
    """count_files' one-pass split-trim-count mode (``adapter``), with the members of :class:`_PlainCount`.
    Set-up errors surface in the order of the two-stage run: every file's split, then the count."""
    line = "{0}: Reads: {1} With barcode and cut site: {2} Clipped on 3' end: {3} With tag: {4}"

    def __init__(self, bckeys, files, rows, tags, cutsite, maxreads, adapter, split_cutsite, split_maxreads):
        from . import hostio, splitter
        if not isinstance(adapter, str) or adapter not in hostio.adapters:
            raise ValueError("unknown adapter set %r (one of %s)" % (adapter, ", ".join(sorted(hostio.adapters))))
        if maxreads != 5e9:
            raise ValueError("maxreads does not apply with adapter: a split file holds at most split_maxreads reads")
        if split_maxreads is None or not float(split_maxreads) <= 5e9:
            raise ValueError("split_maxreads must be at most 5e9, the number of reads the counter takes from a split file")
        self.adapter = hostio.adapters[adapter]
        self.cutsite = hostio.enzymes[adapter[:adapter.find("-")]] if split_cutsite is None else split_cutsite
        for f in files:
            splitter._check_args(self.cutsite, bckeys[f][0], self.adapter)
            splitter._split_patterns(bckeys[f][0], self.cutsite)
        self.plan = matchset.plan([""], tags, cutsite)
        if self.plan.ntags == 0:
            raise IndexError("list index out of range")
        self.tags = self.plan.tags
        self.bckeys, self.rows, self.maxreads = bckeys, rows, split_maxreads

    def whole(self, eng, f, next_file=None):
        """[reads, with barcode and cut site, clipped on the 3' end, with tag] of file ``f``."""
        from . import splitter
        return splitter.count_trimmed_file(eng, f, self.bckeys[f][0], self.rows[f], self.plan, cutsite=self.cutsite,
                                           adapter=self.adapter, maxreads=self.maxreads)

    def own(self, eng, f, rank, dev, n, shard):
        from . import splitter
        start, tail, _first, max_records = shard
        if tail:
            eng.memcpy_h2d(dev + n, np.frombuffer(tail, dtype=np.uint8).ctypes.data, len(tail))
        return splitter.count_trimmed_resident(eng, dev + start, n - start + len(tail), self.bckeys[f][0], self.rows[f],
                                               self.plan, self.cutsite, self.adapter, max_records)


SHARD_MIN_BYTES = 1 << 20     # files smaller than this per rank are not worth cutting up


def shard_files(files, world):
    """The files of a key that count_files cuts into one range per rank (both counting modes), each with
    its BGZF member index (None for a plain file): with fewer files than ranks, every file that is large
    enough and either plain (uncompressed: cut by byte ranges) or a clean BGZF member chain
    (``_native.bgzf_index``: cut by member ranges, which are inflated on the device, so not with
    TDG_GZDEV=0).  The other files are dealt whole to the ranks."""
    if world <= 1 or len(files) >= world:
        return {}
    out = {}
    for f in files:
        if not shardable(f, world):
            continue
        if not _is_gz(f):
            out[f] = None
        elif not _host_inflate_only():
            try:
                index = _native.bgzf_index(f)
            except _native.TdgError:
                index = None
            if index is not None:
                out[f] = index
    return out


def _host_inflate_only():
    """TDG_GZDEV=0, read as the library reads it (atoi): gzip files are inflated on the host."""
    e = os.environ.get("TDG_GZDEV")
    if e is None:
        return False
    m = re.match(r"\s*([+-]?\d+)", e)
    return m is None or int(m.group(1)) == 0


def shardable(f, world):
    try:
        return os.path.getsize(f) >= SHARD_MIN_BYTES * world
    except OSError:
        return False


def range_bounds(path, world):
    """Byte offsets b[0..world] that cut ``path`` into ``world`` ranges of whole lines: b[r] is
    the position after the first '\n' at or beyond r * size / world (b[0] = 0, b[world] = size).
    None when a nominal boundary is followed by no '\n' within 16 MiB (a file with lone-'\r' line
    ends or giant lines: count it on one rank)."""
    size = os.path.getsize(path)
    bounds = [0]
    with open(path, "rb") as fh:
        for r in range(1, world):
            pos = max(bounds[-1], size * r // world)
            fh.seek(pos)
            found = -1
            scanned = 0
            while scanned < (16 << 20):
                block = fh.read(1 << 16)
                if not block:
                    found = size                   # end of file: the tail belongs to the previous range
                    break
                k = block.find(b"\n")
                if k >= 0:
                    found = pos + scanned + k + 1
                    break
                scanned += len(block)
            if found < 0:
                return None
            bounds.append(min(found, size))
    bounds.append(size)
    return bounds


def _device_room(n):
    """The allocation tdg_count_device asks for behind a device image of ``n`` bytes."""
    return (n + _native.TDG_TILE_BYTES - 1) // _native.TDG_TILE_BYTES * _native.TDG_TILE_BYTES + _native.TDG_HALO_BYTES


def _load_range(eng, path, lo, n, extra=0):
    """Bytes [lo, lo + n) of ``path`` in a fresh device allocation padded as tdg_count_device asks, with
    ``extra`` more bytes of room behind them; read with pread through one pinned buffer of at most
    256 MiB.  Returns the device pointer (free with device_free)."""
    dev = eng.device_alloc(_device_room(n + extra))
    try:
        piece = 256 << 20
        host = eng.host_alloc(min(piece, max(n, 1)))
        try:
            view = (ctypes.c_ubyte * min(piece, max(n, 1))).from_address(host)
            with open(path, "rb", buffering=0) as fh:
                done = 0
                while done < n:
                    want = min(piece, n - done)
                    got = os.preadv(fh.fileno(), [memoryview(view)[:want]], lo + done)
                    if got <= 0:
                        raise OSError("short read on " + path)
                    eng.memcpy_h2d(dev + done, host, got)
                    done += got
        finally:
            eng.host_free(host)
    except BaseException:
        eng.device_free(dev)
        raise
    return dev


HEAD_CAP = 1 << 20            # a range whose first three lines are longer than this is not sharded
_TERMINATOR = re.compile(rb"\r\n|\r|\n")


def line_ends(data, k, whole=True):
    """Offsets just past the first ``k`` line terminators of ``data`` (universal newlines: '\\n', '\\r\\n'
    or a lone '\\r'); fewer when there are fewer.  A '\\r' that is the last byte ends a line only when
    ``whole`` (nothing follows data that could make it '\\r\\n')."""
    ends = []
    for m in _TERMINATOR.finditer(data):
        if len(ends) == k or (m.end() == len(data) and m.group() == b"\r" and not whole):
            break
        ends.append(m.end())
    return ends


def range_head(path, lo, hi):
    """The head of the range [lo, hi) of ``path``: its bytes up to and including its third line
    terminator, or all of them when it has fewer.  None when that is longer than HEAD_CAP."""
    with open(path, "rb") as fh:
        fh.seek(lo)
        data = fh.read(min(hi - lo, HEAD_CAP + 1))
    return _head(data, len(data) == hi - lo)


def _device_head(eng, dev, n):
    """:func:`range_head` of the ``n`` bytes of text at device address ``dev``."""
    k = min(n, HEAD_CAP + 1)
    buf = np.empty(k, dtype=np.uint8)
    if k:
        eng.memcpy_d2h(buf.ctypes.data, dev, k)
    return _head(buf.tobytes(), k == n)


def _head(data, whole):
    """The head of a range that begins with ``data`` (all of it when ``whole``)."""
    ends = line_ends(data, 3, whole)
    if len(ends) == 3:
        data = data[:ends[2]]
    elif not whole:
        return None
    return data if len(data) <= HEAD_CAP else None


def plan_trimmed_shards(lines, heads, limit):
    """Lines up the byte ranges of a sharded file on record boundaries, from every range's line starts
    ``lines[k]`` and head ``heads[k]`` (:func:`range_head`).  Records are groups of four lines counted
    from the start of the file, so range k has base_k = sum(lines[:k]) lines before it, and its first
    skip_k = (4 - base_k % 4) % 4 lines finish a record that began before it.  Range k owns its text
    from its first whole record on, plus the first skip_{k+1} lines of range k + 1 (from that range's
    head): whole records, except at the end of the file.

    Returns, per range, (start, tail, first, max_records): the owned text is range[start:] + tail, its
    first record is record ``first`` of the file, and at most max_records = max(0, limit - first) of its
    records are taken (``limit``: the file's record limit, limit_from_maxreads).  None when some range
    holds fewer than skip_k + 1 line starts, or its head fewer than skip_k line ends."""
    skips, firsts, base = [], [], 0
    for k, n in enumerate(lines):
        skip = (4 - base % 4) % 4
        if n < skip + 1 or len(line_ends(heads[k], skip)) < skip:
            return None
        skips.append(skip)
        firsts.append((base + skip) // 4)
        base += n
    out = []
    for k in range(len(lines)):
        start = line_ends(heads[k], skips[k])[-1] if skips[k] else 0
        tail = heads[k + 1][:line_ends(heads[k + 1], skips[k + 1])[-1]] if k + 1 < len(lines) and skips[k + 1] else b""
        out.append((start, tail, firsts[k], max(0, limit - firsts[k])))
    return out


LOOKAHEAD_CAP = 16 << 20     # as range_bounds: a cut followed by no '\n' within this much text is not sharded


def plan_bgzf_share(off, isize, size, rank, world, text_of, cap=None):
    """The text rank ``rank`` of ``world`` owns of a BGZF file of ``size`` bytes whose members start at file
    offsets ``off`` and hold ``isize`` bytes of text each (``_native.bgzf_index``): :func:`range_bounds` in
    text coordinates.  The file is cut at members: c[r] is the first member that starts at or after
    size * r // world (c[0] = 0, c[world] = the end), a function of the file alone, so every rank finds the same
    cuts.  T_r is the text of members [c[r], c[r+1]).  Rank r > 0 owns text from just after the first '\n' of
    T_r; rank r < world - 1 owns text up to just after the first '\n' of T_{r+1}, which it finds by looking
    ahead, member after member, at most ``cap`` bytes of text (LOOKAHEAD_CAP) into T_{r+1}.  So every range
    starts at a line start, and the ranges of all ranks put together are the whole text.

    ``text_of(k0, k1)`` returns the text of members [k0, k1).  Returns (lo, hi, k_first, k_last, front, back):
    the owned text is text[lo:hi] = front + the text of members [k_first, k_last) + back.  None (count the
    file whole) when T_r has no '\n' within ``cap`` bytes (r > 0), the look-ahead finds none within ``cap``
    bytes, or the owned text is empty."""
    cap = LOOKAHEAD_CAP if cap is None else cap
    m = len(off)
    t = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(np.asarray(isize, dtype=np.int64), out=t[1:])
    starts = np.asarray(off, dtype=np.int64)
    c = [0] + [int(np.searchsorted(starts, size * r // world, side="left")) for r in range(1, world)] + [m]

    def first_lf(k, stop):
        """(text of members [k, j), the position of its first '\n') for the first j that holds one; members
        are taken one, two, four ... at a time.  None when members [k, stop) hold none within ``cap`` bytes."""
        got, n, step = [], 0, 1
        while k < stop and n < cap:
            j = min(stop, k + step)
            piece = text_of(k, j)
            at = piece.find(b"\n")
            if at >= 0:
                return (b"".join(got) + piece, n + at, j) if n + at < cap else None
            got.append(piece)
            n += len(piece)
            k, step = j, step * 2
        return None

    lo, k_first, front = 0, 0, b""
    if rank > 0:
        found = first_lf(c[rank], c[rank + 1])
        if found is None:
            return None
        data, at, k_first = found
        lo, front = int(t[c[rank]]) + at + 1, data[at + 1:]
    hi, k_last, back = int(t[m]), m, b""
    if rank < world - 1:
        found = first_lf(c[rank + 1], m)
        if found is None:
            return None
        data, at, _ = found
        hi, k_last, back = int(t[c[rank + 1]]) + at + 1, c[rank + 1], data[:at + 1]
    return (lo, hi, k_first, k_last, front, back) if lo < hi else None


def _load_bgzf_share(eng, path, index, rank, world, extra, ascii_only):
    """The owned text of a BGZF file (:func:`plan_bgzf_share`) in a fresh device allocation padded as
    tdg_count_device asks, with ``extra`` bytes of room behind it: the members in between are inflated on the
    device straight into it (``tdg_bgzf_inflate_device``), the partial members at its two ends, which the
    plan inflated to find the cuts, are copied there from the host.  Returns (device pointer, length), or
    None when the plan refuses, or ``ascii_only`` and a byte of the text is >= 0x80."""
    off, isize = index
    size = os.path.getsize(path)
    t = np.zeros(len(off) + 1, dtype=np.int64)
    np.cumsum(np.asarray(isize, dtype=np.int64), out=t[1:])

    def at(k):
        return int(off[k]) if k < len(off) else size

    def text_of(k0, k1):
        n = int(t[k1] - t[k0])
        if not n:
            return b""
        dev = eng.device_alloc(n)
        try:
            got, _high = eng.bgzf_inflate_device(path, at(k0), at(k1), dev, n)
            buf = np.empty(got, dtype=np.uint8)
            eng.memcpy_d2h(buf.ctypes.data, dev, got)
        finally:
            eng.device_free(dev)
        return buf.tobytes()

    share = plan_bgzf_share(off, isize, size, rank, world, text_of)
    if share is None:
        return None
    lo, hi, k_first, k_last, front, back = share
    if ascii_only and not (front.isascii() and back.isascii()):
        return None
    n = hi - lo
    mid = n - len(front) - len(back)
    dev = eng.device_alloc(_device_room(n + extra))
    try:
        if front:
            eng.memcpy_h2d(dev, np.frombuffer(front, dtype=np.uint8).ctypes.data, len(front))
        if mid:
            got, high = eng.bgzf_inflate_device(path, at(k_first), at(k_last), dev + len(front), mid)
            if got != mid:
                raise _native.TdgError(_native.TDG_ERR_GZIP, "%s: %d bytes of text where the index has %d" % (path, got, mid))
            if ascii_only and high:
                eng.device_free(dev)
                return None
        if back:
            eng.memcpy_h2d(dev + n - len(back), np.frombuffer(back, dtype=np.uint8).ctypes.data, len(back))
    except BaseException:
        eng.device_free(dev)
        raise
    return dev, n


def _load_share(eng, mode, path, rank, world, index):
    """Step 1 of :func:`_count_sharded` up to the line count: this rank's text of ``path`` in device memory, with
    ``mode.extra`` bytes of room behind it -- its byte range of a plain file (``index`` None: :func:`range_bounds`,
    :func:`_load_range`) or its owned text of a BGZF file (``index``: :func:`_load_bgzf_share`) -- and
    ``mode.payload`` of its head.  Returns (device pointer, length, payload), or None: the rank votes for
    counting the file whole."""
    if index is None:
        bounds = range_bounds(path, world)
        if bounds is None or bounds[rank] >= bounds[rank + 1]:
            return None
        lo, hi = bounds[rank], bounds[rank + 1]
        payload = mode.payload(lambda: range_head(path, lo, hi))
        if payload is None:
            return None
        return _load_range(eng, path, lo, hi - lo, extra=mode.extra), hi - lo, payload
    loaded = _load_bgzf_share(eng, path, index, rank, world, mode.extra, mode.ascii_only)
    if loaded is None:
        return None
    dev, n = loaded
    try:
        payload = mode.payload(lambda: _device_head(eng, dev, n))
    except BaseException:
        eng.device_free(dev)
        raise
    if payload is None:
        eng.device_free(dev)
        return None
    return dev, n, payload


def _place_share(eng, mode, path, rank, world, gather, index=None):
    """Steps 1 to 3 of :func:`_count_sharded`, which :func:`splitter.split_files` shares: this rank's text of
    ``path`` loaded (``mode.extra`` bytes of room behind it), its line starts counted, the first ``gather``
    and ``mode.place``.  Returns (device pointer, length, share), or None on every rank when the file is to
    be handled whole by rank 0 (nothing is left allocated then)."""
    if gather is None:
        raise ValueError("sharding a file across ranks needs a gather callable (see dist_gather)")
    dev, n, lines, payload = None, 0, 0, None
    try:
        loaded = _load_share(eng, mode, path, rank, world, index)
        if loaded is not None:
            dev, n, payload = loaded
            lines, _last = eng.count_lines_device(dev, n, 0, _native.TDG_PREV_NONE if rank == 0 else _native.TDG_PREV_LF)
    except (OSError, _native.TdgError):
        if dev is not None:
            eng.device_free(dev)
            dev = None                          # this rank votes for handling the file whole
    every = gather([0] if dev is None else [1, lines] + payload)
    share = None
    if all(x[0] for x in every):
        share = mode.place([x[1] for x in every], [x[2:] for x in every], rank)
    if share is None:
        if dev is not None:
            eng.device_free(dev)
        return None
    return dev, n, share


def _gather_checked(gather, path, err, values, doing):
    """A ``gather`` of [failed, values...] after a step every rank ran on its own share: raises ``err`` on the
    rank that failed, a RuntimeError naming the first failed rank on the others.  Returns every rank's values."""
    every = gather([0 if err is None else 1] + list(values))
    if err is not None:
        raise err
    failed = [k for k, x in enumerate(every) if x[0]]
    if failed:
        raise RuntimeError("%s: rank %d failed while %s its byte range" % (path, failed[0], doing))
    return [x[1:] for x in every]


def _count_sharded(eng, mode, path, rank, world, gather, index=None):
    """One file that count_files cuts into one range per rank (:func:`shard_files`), in either counting
    mode (``mode``: :class:`_PlainCount` or :class:`_TrimmedCount`); ``index``: the member index of a BGZF
    file, None for a plain file.  Lines, reads and records are numbered from the start of the FILE
    (tagdigger_fun.py:250-254), so a range cannot be counted on its own:

    1. every rank loads its range into device memory (:func:`_load_share`: a byte range of a plain file, the
       owned text of a BGZF file, inflated on the device), with ``mode.extra`` bytes of room behind it, and
       counts its line starts there (``tdg_count_lines_device``);
    2. one ``gather`` of [ok, line starts, ``mode.payload``] tells every rank where its range lies in the
       file (``mode.place``);
    3. if some rank cannot take part (no cut point or an empty range, a failed load or inflate, no payload,
       a byte >= 0x80 in BGZF text of the plain mode) or
       ``mode.place`` refuses, rank 0 counts the file whole (``mode.whole``), exactly as a file dealt whole:
       nothing has touched the matrix yet;
    (steps 1 to 3 are :func:`_place_share`)
    4. otherwise every rank counts its range (``mode.own``);
    5. a second ``gather`` of [failed, totals] sums the totals.  A rank that failed in step 4 raises its
       own exception after that gather, the others a RuntimeError naming it.

    Returns the file's totals, or None on the ranks other than 0 when rank 0 counted the file whole."""
    placed = _place_share(eng, mode, path, rank, world, gather, index)
    if placed is None:
        return mode.whole(eng, path) if rank == 0 else None
    dev, n, share = placed
    tot, err = [], None
    try:
        tot = mode.own(eng, path, rank, dev, n, share)
    except Exception as e:                      # every rank still takes part in the second gather
        err = e
    finally:
        eng.device_free(dev)
    every = _gather_checked(gather, path, err, [int(t) for t in tot], "counting")
    return [sum(t) for t in zip(*every)]


def dist_gather(values):
    """all_gather of a short list of ints over the default torch.distributed group."""
    import torch.distributed as dist
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, list(values))
    return out


def assign_files(files, rank, world):
    """The files rank ``rank`` of ``world`` counts: longest-processing-time-first
    by file size, ties and unreadable sizes in name order (deterministic on every
    rank)."""
    if world <= 1:
        return list(files)

    def size(f):
        try:
            return os.path.getsize(f)
        except OSError:
            return 0
    load = [0] * world
    mine = []
    for f in sorted(files, key=lambda f: (-size(f), f)):
        r = min(range(world), key=lambda k: (load[k], k))
        load[r] += max(size(f), 1)
        if r == rank:
            mine.append(f)
    return sorted(mine)


def nccl_reduce(ptr, rows, cols, eng):
    """Sum the per-GPU count matrices in place with ONE all-reduce, issued in
    stream order behind the last count kernel (the multi-GPU form of the sum in
    combineReadCounts, tagdigger_fun.py:1088-1095).  Needs an initialised
    torch.distributed process group (backend nccl)."""
    import torch
    import torch.distributed as dist

    class _View(object):          # the library's matrix as a torch tensor, without copying
        pass
    v = _View()
    v.__cuda_array_interface__ = {"shape": (rows, cols), "typestr": "<i4", "data": (ptr, False), "version": 3,
                                  "strides": None}
    t = torch.as_tensor(v, device=torch.device("cuda", eng.device))
    stream = torch.cuda.current_stream().cuda_stream
    eng.other_stream_wait(stream)
    dist.all_reduce(t)
    eng.stream_wait(stream)


def init_comm(eng, rank, world):
    """Give the engine its own NCCL communicator (``tdg_comm_init``): rank 0 makes the id, the
    default torch.distributed group (any backend) carries the 128 bytes to the other ranks."""
    import torch.distributed as dist
    ids = [eng.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    eng.comm_init(ids[0], world, rank)


def engine_reduce(ptr, rows, cols, eng):
    """``reduce`` for :func:`count_files`: the library's own all-reduce on the counting stream
    (``tdg_allreduce_matrix``; needs :func:`init_comm` first).  No torch tensor is involved."""
    eng.allreduce_matrix()
