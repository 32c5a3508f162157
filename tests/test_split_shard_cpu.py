"""The output of one library file that split_files shards across ranks, checked without a GPU: the file is
cut at range_bounds, every range is placed with counting.plan_trimmed_shards, the oracle's barcodeSplitter
loop runs over each rank's owned text (with that rank's max_records), and each rank's bytes are put at the
offsets splitter.shard_offsets gives.  The output files must equal the oracle's whole-file files byte for
byte, and the progress lines composed from each rank's flags and prefix totals must equal the whole-file
run's lines."""

import io
import random

import numpy as np
import pytest

from helpers import rand_seq
from oracle import tagdigger_oracle as orc
from tagdigger_b200 import _native, counting, hostio, splitter

BARCODES = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA", "AACCGT"]
ADAPTER = hostio.adapters["PstI-MspI-Hall"]
SITE = "TGCAG"
NAME = "lib.fq"


@pytest.fixture(scope="module")
def library():
    """About 120,000 short records: barcode + cut site + insert, some running into the adapter or the
    common-cutter site, some without a barcode, some lower case or with blanks."""
    rng = random.Random(11)
    a0 = ADAPTER[0][0].replace("^", "") + ADAPTER[0][1]
    out = []
    for i in range(120000):
        bc = rng.choice(BARCODES) if rng.random() < 0.9 else rand_seq(rng, 5)
        s = bc + SITE + rand_seq(rng, rng.randint(0, 25))
        k = rng.random()
        if k < 0.3:
            s += a0[:rng.randint(1, 20)]
        elif k < 0.4:
            s += "CCGG" + rand_seq(rng, 5)
        if k > 0.95:
            s = s.lower()
        elif k > 0.92:
            s = " " + s + "\t"
        q = "".join(rng.choice("ABCDEFGHIJ#") for _ in range(len(s.strip())))
        out.append("@r%d\n%s\n%s\n%s\n" % (i, s, "+" if rng.random() < 0.8 else "+r%d" % i, q))
    return "".join(out)


def oracle_split(text, maxreads):
    """barcodeSplitter over ``text`` per the oracle: (bytes of every barcode's file, flags per record,
    progress lines as the reference prints them)."""
    bufs = [io.StringIO() for _ in BARCODES]
    flags, lines, c = [], [], [0, 0, 0]
    for b, recs, s2 in orc.split_records(io.StringIO(text, newline=None), BARCODES, SITE, ADAPTER, maxreads, every=True):
        f = 0
        if b > -1:
            f = 1 | (2 if s2 != 999 else 0)
            bufs[b].write("".join(ln + "\n" for ln in recs))
        flags.append(f)
        c = [c[0] + 1, c[1] + (f & 1), c[2] + (f >> 1)]
        if c[0] % 1000000 == 0:
            lines.append(NAME)
        if c[0] % 50000 == 0:
            lines.append("Reads: {0} With barcode and cut site: {1} Clipped on 3' end: {2}".format(*c))
    return [b.getvalue().encode("utf-8") for b in bufs], np.asarray(flags, dtype=np.uint8), lines


_whole = {}


def whole(text, maxreads):
    key = (text, maxreads)
    if key not in _whole:
        _whole.clear()
        _whole[key] = oracle_split(text, maxreads)
    return _whole[key]


def line_starts(data):
    return len(io.StringIO(data.decode("utf-8"), newline=None).readlines())


def check(tmp_path, text, world, maxreads=500000000):
    """The ranks' bytes at their offsets are the whole-file files, their lines the whole-file lines.
    Returns the shards."""
    path = tmp_path / NAME
    path.write_bytes(text.encode("utf-8"))
    data = path.read_bytes()
    bounds = counting.range_bounds(str(path), world)
    assert bounds is not None
    spans = list(zip(bounds[:-1], bounds[1:]))
    lines = [line_starts(data[lo:hi]) for lo, hi in spans]
    heads = [counting.range_head(str(path), lo, hi) for lo, hi in spans]
    shards = counting.plan_trimmed_shards(lines, heads, _native.limit_from_maxreads(maxreads))
    assert shards is not None, (world, bounds)
    runs = []
    for k, (start, tail, _first, max_records) in enumerate(shards):
        if max_records == 0:
            runs.append(([b""] * len(BARCODES), np.zeros(0, dtype=np.uint8)))
            continue
        owned = data[bounds[k] + start:bounds[k + 1]] + tail
        files, flags, _lines = oracle_split(owned.decode("utf-8"), max_records)
        runs.append((files, flags))
    sizes = [[len(f) for f in files] for files, _ in runs]
    totals = [[len(fl), int(np.count_nonzero(fl & 1)), int(np.count_nonzero(fl & 2))] for _, fl in runs]
    want_files, want_flags, want_lines = whole(text, maxreads)
    assert sum(t[0] for t in totals) == len(want_flags)
    got = [bytearray(sum(s[b] for s in sizes)) for b in range(len(BARCODES))]
    out = []
    for k, (files, flags) in enumerate(runs):
        offsets = splitter.shard_offsets(sizes, k)
        for b, piece in enumerate(files):
            got[b][offsets[b]:offsets[b] + len(piece)] = piece
        splitter._Progress(NAME, splitter.shard_offsets(totals, k), out.append).many(flags)
    for b in range(len(BARCODES)):
        assert bytes(got[b]) == want_files[b], (world, b)
    assert out == want_lines, world
    return shards


def shifted_at_cuts(text, world):
    """A blank line right after the first line end at or past every nominal cut."""
    data = text.encode("utf-8")
    out = bytearray(data)
    for r in reversed(range(1, world)):
        pos = data.index(b"\n", len(data) * r // world) + 1
        out[pos:pos] = b"\n"
    return out.decode("utf-8")


def landing_line(text, world):
    data = text.encode("utf-8")
    return (line_starts(data[:len(data) // world + 1]) - 1) % 4


@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_sharded_split_equals_whole_file(tmp_path, library, world):
    text = library
    shards = check(tmp_path, text, world)
    assert shards[0][2] == 0 and all(s[3] > 0 for s in shards)
    for t in (text.replace("\n", "\r\n"), shifted_at_cuts(text, world), text[:-1], text + "@x\nACGTATGCAGTT\n",
              text + "@x\nACGTATGCAGTT"):
        check(tmp_path, t, world)


def test_progress_lines_fall_in_different_ranks(tmp_path, library):
    _files, _flags, lines = whole(library, 500000000)
    assert len(lines) == 2
    shards = check(tmp_path, library, 2)
    assert shards[1][2] < 100000 and shards[1][2] > 50000


def test_cut_in_each_line_of_a_record(tmp_path, library):
    """The first cut of world 2 falls in each of a record's four lines (a longer first header moves it)."""
    hits = {}
    for pad in range(400):
        t = "@pad" + "x" * pad + library[library.index("\n"):]
        hits.setdefault(landing_line(t, 2), t)
        if len(hits) == 4:
            break
    assert sorted(hits) == [0, 1, 2, 3]
    for t in hits.values():
        check(tmp_path, t, 2)


def test_maxreads_inside_and_at_rank_1(tmp_path, library):
    shards = check(tmp_path, library, 3)
    first = shards[1][2]
    sh = check(tmp_path, library, 3, maxreads=first + 5000)
    assert sh[1][3] == 5000 and sh[2][3] == 0
    sh = check(tmp_path, library, 3, maxreads=first)
    assert sh[1][3] == 0 and sh[2][3] == 0


def test_shard_offsets():
    assert splitter.shard_offsets([[3, 0, 5], [1, 2, 0], [4, 4, 4]], 0) == [0, 0, 0]
    assert splitter.shard_offsets([[3, 0, 5], [1, 2, 0], [4, 4, 4]], 2) == [4, 2, 5]
    assert splitter.shard_offsets([[3, 0, 5], [1, 2, 0], [4, 4, 4]], 3) == [8, 6, 9]
