"""Host side of the counting path: the drop-in for ``find_tags_fastq``.

Mirrors /root/reference/tagdigger_fun.py:192-277 (same signature, defaults,
asserts and return shape); the per-read loop runs on the GPU through
``_native.Engine`` (ctypes over include/tagdigger_b200.h).  Nothing here counts
reads on the CPU.
"""

import ctypes
import gzip
import os
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
        if e.code == _native.TDG_ERR_GZIP:
            raise _gzip_exception(e.message)
        if e.code == _native.TDG_ERR_IO:
            raise OSError(e.message)
        if e.code == _native.TDG_ERR_UTF8:
            # open(f, 'r') / gzip.open(f, 'rt') decode the file as UTF-8 (tagdigger_fun.py:240-243)
            pos = int(e.message.split()[1].rstrip(":")) if e.message.startswith("position ") else 0
            raise UnicodeDecodeError("utf-8", b"\xff", 0, 1, "invalid UTF-8 at byte %d (%s)" % (pos, e.message))
        raise


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
    fewer files than ranks, plain files are sharded by byte range instead (:func:`count_file_range`),
    which needs ``gather(list_of_ints) -> list of every rank's list`` (:func:`dist_gather`).

    Returns ``[sample names, count rows]`` -- rows as lists of int like combineReadCounts, or,
    with ``as_array=True``, as one int32 ndarray (hostio.writeCounts / writeDiploidGeno format
    that with native threads; a 384 x 500,000 matrix is 768 MB as an array and several GB as
    Python integers).  ``totals`` (optional dict) receives ``{file: [reads, with barcode and
    cut site, with tag]}`` for this rank's files.

    With ``adapter`` (the name of an adapter set, a key of ``hostio.adapters``) every file is first
    split and trimmed as ``barcodeSplitter(f, barcodes, files, cutsite=split_cutsite, adapter=...,
    maxreads=split_maxreads)`` would, and each barcode's output is then counted as
    ``find_tags_fastq(file, [''], tags, cutsite)`` into its sample's row -- in one pass per file on the
    GPU, without writing the split files (:func:`splitter.count_trimmed_file`).  ``split_cutsite``
    defaults to the cut site of the adapter set's enzyme, as barcode_splitter_script derives it.  Files
    are dealt whole to the ranks.  ``totals`` then receives ``[reads, with barcode and cut site, clipped
    on the 3' end, with tag]``."""
    files = sorted(bckeys.keys())
    samples, rows = global_rows(bckeys)
    if adapter is not None:
        eng = _count_trimmed_files(bckeys, files, rows, len(samples), tags, cutsite, maxreads, device, rank, world,
                                   totals, adapter, split_cutsite, split_maxreads)
        return _result(eng, samples, len(tags), world, reduce, as_array)
    limit = _native.limit_from_maxreads(maxreads)
    plans = {}
    tagplan = None
    for f in files:                               # set-up errors surface before any counting, file by file
        if tagplan is None:
            plans[f] = matchset.plan(bckeys[f][0], tags, cutsite)
            tagplan = matchset.plan_tags(tags, cutsite)       # shared by the other files of the key
        else:
            plans[f] = matchset.plan(bckeys[f][0], tags, cutsite, tagplan=tagplan)
        if plans[f].barnum == 0 or plans[f].ntags == 0:
            raise IndexError("list index out of range")
    ntags = len(tags)
    eng = get_engine(device)
    first = plans[files[0]]
    eng.set_tags(first.tags.patterns, first.tags.index, any_base=first.tags.any_base)
    eng.set_matrix(len(samples), ntags)
    # Fewer files than GPUs: a plain (uncompressed) file is cut into one byte range per rank
    # (cut at line ends); otherwise whole files are dealt to the ranks.
    split = [f for f in files if world > 1 and len(files) < world and not _is_gz(f) and shardable(f, world)]
    for f in split:
        load_plan(eng, plans[f], row_of=rows[f], set_tags=False)
        tot = count_file_range(eng, f, rank, world, limit, gather)
        if totals is not None:
            totals[f] = tot[:3]
    mine = assign_files([f for f in files if f not in split], rank, world)
    for i, f in enumerate(mine):
        p = plans[f]
        load_plan(eng, p, row_of=rows[f], set_tags=False)
        tot = _run_file(eng, f, limit, next_file=mine[i + 1] if i + 1 < len(mine) else None)
        print("{0}: Reads: {1} With barcode and cut site: {2} With tag: {3}".format(f, tot[0], tot[1], tot[2]))
        if totals is not None:
            totals[f] = tot[:3]
    return _result(eng, samples, ntags, world, reduce, as_array)


def _result(eng, samples, ntags, world, reduce, as_array):
    """count_files' return value: the matrix, summed over the ranks."""
    if world > 1:
        if reduce is None:
            raise ValueError("count_files with world > 1 needs a reduce callable (see nccl_reduce)")
        reduce(eng.matrix_ptr(), len(samples), ntags, eng)
    matrix = eng.read_matrix()
    return [samples, matrix if as_array else matrix.tolist()]


def _count_trimmed_files(bckeys, files, rows, nrows, tags, cutsite, maxreads, device, rank, world, totals, adapter,
                         split_cutsite, split_maxreads):
    """count_files with ``adapter``: this rank's files through splitter.count_trimmed_file.  Returns the engine."""
    from . import hostio, splitter
    if not isinstance(adapter, str) or adapter not in hostio.adapters:
        raise ValueError("unknown adapter set %r (one of %s)" % (adapter, ", ".join(sorted(hostio.adapters))))
    if maxreads != 5e9:
        raise ValueError("maxreads does not apply with adapter: a split file holds at most split_maxreads reads")
    if split_maxreads is None or not float(split_maxreads) <= 5e9:
        raise ValueError("split_maxreads must be at most 5e9, the number of reads the counter takes from a split file")
    adapter_seqs = hostio.adapters[adapter]
    if split_cutsite is None:
        split_cutsite = hostio.enzymes[adapter[:adapter.find("-")]]
    # set-up errors surface before any counting, in the order of the two-stage run: every file's split, then the count
    for f in files:
        splitter._check_args(split_cutsite, bckeys[f][0], adapter_seqs)
        splitter._split_patterns(bckeys[f][0], split_cutsite)
    plan = matchset.plan([""], tags, cutsite)
    if plan.ntags == 0:
        raise IndexError("list index out of range")
    eng = get_engine(device)
    eng.set_tags(plan.tags.patterns, plan.tags.index, any_base=plan.tags.any_base)
    eng.set_matrix(nrows, plan.ntags)
    for f in assign_files(files, rank, world):
        tot = splitter.count_trimmed_file(eng, f, bckeys[f][0], rows[f], plan, cutsite=split_cutsite, adapter=adapter_seqs,
                                          maxreads=split_maxreads)
        print("{0}: Reads: {1} With barcode and cut site: {2} Clipped on 3' end: {3} With tag: {4}".format(f, *tot))
        if totals is not None:
            totals[f] = tot
    return eng


SHARD_MIN_BYTES = 1 << 20     # files smaller than this per rank are not worth cutting up


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


def count_file_range(eng, path, rank, world, limit, gather):
    """One rank's share of a plain FASTQ file that is sharded across ``world`` GPUs.

    The file is cut at line ends into one byte range per rank.  Which lines are sequence lines
    depends on the line index from the start of the FILE (tagdigger_fun.py:250-254), so every
    rank first counts the lines of its range on its GPU (``tdg_count_lines_device``: the scan
    half of the kernel), the counts are exchanged (``gather``), and the range is then counted
    with its true first line index (``tdg_count_device``).  ``maxreads`` works unchanged: read
    indices are global.  Returns this rank's [reads, with barcode and cut site, with tag]."""
    if gather is None:
        raise ValueError("sharding a file across ranks needs a gather callable (see dist_gather)")
    bounds = range_bounds(path, world)
    ok = gather([0 if bounds is None else 1])
    if not all(x[0] for x in ok):                       # every rank must take the same decision
        bounds = None
    if bounds is None:
        tot = [0, 0, 0, 0]
        if rank == 0:
            tot = _run_file(eng, path, limit)
        return tot
    lo, hi = bounds[rank], bounds[rank + 1]
    n = hi - lo
    cap = (n + _native.TDG_TILE_BYTES - 1) // _native.TDG_TILE_BYTES * _native.TDG_TILE_BYTES + _native.TDG_HALO_BYTES
    dev = eng.device_alloc(cap)
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
        lines, _last = eng.count_lines_device(dev, n, 0, _native.TDG_PREV_NONE if rank == 0 else _native.TDG_PREV_LF)
        every = gather([lines])
        base = sum(x[0] for x in every[:rank])
        eng.reset_file()
        eng.count_device(dev, n, base, _native.TDG_PREV_NONE if rank == 0 else _native.TDG_PREV_LF, limit)
        tot = eng.file_totals()
    finally:
        eng.device_free(dev)
    print("{0} [bytes {1}-{2}]: Reads: {3} With barcode and cut site: {4} With tag: {5}".format(path, lo, hi, *tot[:3]))
    return tot


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
