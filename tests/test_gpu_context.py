"""The context's buffers and events (csrc/tdg_api.cu): an allocation that fails anywhere leaves a
context that works.  TDG_FAIL_ALLOC=k makes the k-th buffer allocation or event creation of an engine
fail with TDG_ERR_NOMEM; the call reports it, the same calls made again succeed, and every result
equals that of a run without a failure."""

import contextlib
import gzip
import io
import random

import numpy as np
import pytest

from feed_check import bgzf_compress
from tagdigger_b200 import _native, hostio, matchset, synth, trimming

pytestmark = pytest.mark.gpu

CHUNK = 1 << 20
BOUND = 300              # allocations and event creations of the whole sequence, both passes


class Inputs:
    """Tables and text of one pass.  The second pass is larger in every table and input, so that its
    allocations are regrowths of the first pass's buffers."""

    def __init__(self, tmp_path, big):
        rng = np.random.default_rng(31 + big)
        r = random.Random(17 + big)
        nbar, npairs, nreads = (12, 300, 6000) if big else (4, 40, 1500)
        self.barcodes = synth.make_barcodes(nbar, rng)
        _, _, seqs = synth.make_marker_pairs(npairs, rng)
        tags = [s for p in seqs for s in p]
        self.fq, _ = synth.make_fastq(nreads, self.barcodes, tags, rng)
        self.plan = matchset.plan(self.barcodes, tags, "TGCAG")
        self.plain = str(tmp_path / ("reads%d.fq" % big))
        self.gz = str(tmp_path / ("reads%d.fq.gz" % big))
        with open(self.plain, "wb") as fh:
            fh.write(self.fq)
        with open(self.gz, "wb") as fh:
            fh.write(gzip.compress(self.fq, 6))
        self.bgzf = str(tmp_path / ("reads%d.bgzf.gz" % big))
        with open(self.bgzf, "wb") as fh:
            fh.write(bgzf_compress(self.fq))
        barcut = hostio.combine_barcode_and_cutsite(self.barcodes, "TGCAG")
        self.split_bar = matchset.effective_set(barcut, len(barcut))
        with contextlib.redirect_stdout(io.StringIO()):
            self.trim = trimming.trim_tables(hostio.adapters["PstI-MspI-Hall"], self.barcodes)
        self.seqs = self.fq.split(b"\n")[1::4]
        self.bars = [r.randrange(nbar) for _ in self.seqs]
        self.starts = [r.randrange(12) for _ in self.seqs]
        self.tails = [(b"@extra %d\nACGT\n+\nIIII\n" % b) * (300 + 50 * b) for b in range(nbar)]


# ---- the units: each starts from its own set-up call, so that it can be run again after a failure.
# A unit returns (result, feed): result must equal the failure-free run's, feed is how a gzip file was fed.

def _tables(eng, d):
    p = d.plan
    eng.set_tags(p.tags.patterns, p.tags.index, any_base=p.tags.any_base)
    eng.set_matrix(p.barnum, p.ntags)
    return None, None


def _begin(eng, d):
    p = d.plan
    eng.zero_matrix()
    eng.begin_file(p.bar.patterns, p.bar.index, p.bar_tag_off, any_base=p.bar.any_base)


def _submit(eng, d):
    _begin(eng, d)
    eng.submit(d.fq)
    eng.end_file()
    return (eng.read_matrix().tobytes(), eng.file_totals()), None


def _count(eng, path):
    tot = eng.count_file(path, path.endswith(".gz"))
    return (eng.read_matrix().tobytes(), tot), eng.last_file_info()["mode"]


def _plain_file(eng, d):
    _begin(eng, d)
    return _count(eng, d.plain)


def _gzip_file(eng, d):
    _begin(eng, d)
    return _count(eng, d.gz)


def _bgzf_file(eng, d):
    _begin(eng, d)
    return _count(eng, d.bgzf)


def _released_gzip_file(eng, d):
    eng.release_scratch()
    return _gzip_file(eng, d)


def _timed(eng, d):
    eng.timing_begin()
    _begin(eng, d)
    out, _ = _count(eng, d.plain)
    ms, timed = eng.timing_end()
    return (out, timed), None


def _trim(eng, d):
    eng.set_trim(*d.trim)
    return eng.trim_batch(d.seqs, d.bars, d.starts), None


def _split(eng, d):
    b = d.split_bar
    eng.begin_file(b.patterns, b.index, [len(x) for x in b.patterns], any_base=b.any_base)
    eng.split_begin(d.barcodes, 5)
    eng.split_bgzf(True)
    files = [bytearray() for _ in d.barcodes]
    flags = []
    text = np.frombuffer(d.fq, dtype=np.uint8)
    pos = 0
    while pos < len(text):
        n = min(300000, len(text) - pos)
        nrec, used, needs_host, pieces, fl = eng.split_block(text.ctypes.data + pos, n, pos + n == len(text), 1 << 40)
        if nrec == 0:
            break
        if needs_host:                                      # (records the splitter leaves to the host)
            flags.append((nrec, used))
        else:
            for f, piece in zip(files, pieces):
                f += bytes(piece)
            flags.append(bytes(fl))
        pos += used
    for f, piece in zip(files, eng.bgzf_append(d.tails)):
        f += bytes(piece)
    for f, piece in zip(files, eng.bgzf_finish()):
        f += bytes(piece)
    return ([bytes(f) for f in files], flags), None


def _split_batch(eng, d):
    bar, cut = eng.split_batch(d.seqs, [len(b) for b in d.barcodes], 5)
    return (bar.tobytes(), cut.tobytes()), None


def _match_batch(eng, d):
    row, col = eng.match_batch(d.seqs)
    return (row.tobytes(), col.tobytes()), None


GZIP_UNITS = (_gzip_file, _bgzf_file, _released_gzip_file)
UNITS = [_tables, _submit, _plain_file, _gzip_file, _bgzf_file, _released_gzip_file, _timed, _trim, _split, _split_batch, _match_batch]


def _sequence(eng, passes):
    """Every unit of both passes.  A unit that fails with TDG_ERR_NOMEM runs once more.
    Returns (results, feeds, whether a simulated failure was met)."""
    results, feeds, failed = [], [], False
    for d in passes:
        for unit in UNITS:
            try:
                out = unit(eng, d)
            except _native.TdgError as e:
                assert e.code == _native.TDG_ERR_NOMEM and "simulated" in e.message, (unit.__name__, e.code, e.message)
                failed = True
                out = unit(eng, d)
            results.append(out[0])
            feeds.append(out[1])
    return results, feeds, failed


def test_allocation_failure_leaves_a_working_context(tmp_path, monkeypatch):
    monkeypatch.setenv("TDG_GZDEV_MIN", "0")                # the device gzip feed takes the small files too
    monkeypatch.delenv("TDG_FAIL_ALLOC", raising=False)
    passes = [Inputs(tmp_path, False), Inputs(tmp_path, True)]
    eng = _native.Engine(0, chunk_bytes=CHUNK)
    want, want_feeds, failed = _sequence(eng, passes)
    eng.close()
    assert not failed
    assert all(want_feeds[UNITS.index(u)] == 0 for u in GZIP_UNITS)

    for k in range(1, BOUND + 1):
        monkeypatch.setenv("TDG_FAIL_ALLOC", str(k))
        eng = _native.Engine(0, chunk_bytes=CHUNK)
        got, feeds, failed = _sequence(eng, passes)
        eng.close()
        for i, (a, b) in enumerate(zip(got, want)):
            assert a == b, "allocation %d: unit %s of pass %d" % (k, UNITS[i % len(UNITS)].__name__, i // len(UNITS))
        handed_over = [i for i, (f, w) in enumerate(zip(feeds, want_feeds)) if f != w]
        assert all(UNITS[i % len(UNITS)] in GZIP_UNITS and feeds[i] == 1 for i in handed_over), (k, feeds)
        if not failed and not handed_over:
            break                                           # k is past the last allocation of the sequence
    else:
        pytest.fail("every one of %d runs met a simulated failure" % BOUND)
    assert k > 50, k                                        # the hook fired in the runs before
