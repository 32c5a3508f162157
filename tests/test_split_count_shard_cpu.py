"""The record alignment of a file that count_files(..., adapter=...) shards across ranks, checked
without a GPU: the file is cut at range_bounds, every range's line starts and head go through
counting.plan_trimmed_shards, and the oracle's two-stage run over each rank's owned text (with that
rank's max_records) must sum to the two-stage run over the whole file, matrix and totals."""

import io
import random

import numpy as np
import pytest

from split_count_check import make_reads, make_tags, two_stage
from tagdigger_b200 import _native, counting, hostio

BARCODES = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA", "AACCGT"]
KEY = {"lib.fq": [BARCODES, ["A", "B", "C", "A", "D"]]}
ADAPTER = hostio.adapters["PstI-MspI-Hall"]


@pytest.fixture(scope="module")
def library():
    rng = random.Random(5)
    tags = make_tags(rng, "TGCAG", 40)
    return tags, make_reads(rng, BARCODES, "TGCAG", tags, ADAPTER, 240)


def line_starts(data):
    return len(io.StringIO(data.decode("utf-8"), newline=None).readlines())


def shard(path, world, maxreads):
    """(bounds, shards) of the sharded count; shards is None when rank 0 counts the file whole."""
    bounds = counting.range_bounds(str(path), world)
    if bounds is None:
        return None, None
    data = path.read_bytes()
    lines = [line_starts(data[lo:hi]) for lo, hi in zip(bounds[:-1], bounds[1:])]
    heads = [counting.range_head(str(path), lo, hi) for lo, hi in zip(bounds[:-1], bounds[1:])]
    if any(h is None for h in heads):
        return bounds, None
    return bounds, counting.plan_trimmed_shards(lines, heads, _native.limit_from_maxreads(maxreads))


def check_sum(tmp_path, text, tags, world, maxreads=500000000):
    """The owned texts of all ranks count to what the whole file counts.  Returns (bounds, shards)."""
    path = tmp_path / "lib.fq"
    path.write_bytes(text.encode("utf-8"))
    bounds, shards = shard(path, world, maxreads)
    assert shards is not None, (world, bounds)
    data = path.read_bytes()
    samples, want, want_tot = two_stage({"lib.fq": text}, KEY, tags, "TGCAG", ADAPTER, "TGCAG", maxreads)
    got = np.zeros((len(samples), len(tags)), dtype=np.int64)
    got_tot = [0, 0, 0, 0]
    for k, (start, tail, _first, max_records) in enumerate(shards):
        if max_records == 0:
            continue
        owned = data[bounds[k] + start:bounds[k + 1]] + tail
        s, m, t = two_stage({"lib.fq": owned.decode("utf-8")}, KEY, tags, "TGCAG", ADAPTER, "TGCAG", max_records)
        assert s == samples
        got += np.asarray(m, dtype=np.int64).reshape(got.shape)
        got_tot = [a + b for a, b in zip(got_tot, t["lib.fq"])]
    assert got.tolist() == np.asarray(want, dtype=np.int64).reshape(got.shape).tolist(), world
    assert got_tot == want_tot["lib.fq"], world
    return bounds, shards


def records(text, newline="\n"):
    lines = text.split(newline)
    return [newline.join(lines[i:i + 4]) + newline for i in range(0, len(lines) - 1, 4)]


def landing_line(text, world):
    """The line index mod 4 of the line the first nominal cut (size / world) falls in."""
    data = text.encode("utf-8")
    return (line_starts(data[:len(data) // world + 1]) - 1) % 4


@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_owned_texts_sum_to_the_file(tmp_path, library, world):
    tags, text = library
    shapes = [("lf", text), ("crlf", text.replace("\n", "\r\n")), ("no final newline", text[:-1]),
              ("partial record", text + "@x\nACGTATGCAGTT\n"),
              ("partial record, no final newline", text + "@x\nACGTATGCAGTT")]
    # a blank line at every nominal cut: the record phase shifts right where a range starts
    data = text.encode("utf-8")
    shifted = bytearray(data)
    for r in reversed(range(1, world)):
        pos = data.index(b"\n", len(data) * r // world) + 1
        shifted[pos:pos] = b"\n"
    shapes.append(("blank line at the cuts", shifted.decode("utf-8")))
    for label, t in shapes:
        bounds, shards = check_sum(tmp_path, t, tags, world)
        assert shards[0][0] == 0 and shards[0][2] == 0, label
    # the first cut falls in each of a record's four lines (a longer first header moves it)
    hits = {}
    for pad in range(400):
        t = "@pad" + "x" * pad + text[text.index(" "):]
        hits.setdefault(landing_line(t, world), t)
    assert sorted(hits) == [0, 1, 2, 3]
    for t in hits.values():
        check_sum(tmp_path, t, tags, world)


def test_maxreads_inside_and_at_a_range(tmp_path, library):
    tags, text = library
    bounds, shards = check_sum(tmp_path, text, tags, 3)
    first = shards[1][2]
    assert 0 < first < shards[2][2]
    for m in (first + 7, first, first - 1, 1, 1.5, shards[2][2] + 3):
        _, sh = check_sum(tmp_path, text, tags, 3, maxreads=m)
        assert sh[1][3] == max(0, _native.limit_from_maxreads(m) - first)
    _, sh = check_sum(tmp_path, text, tags, 3, maxreads=first)
    assert sh[1][3] == 0 and sh[2][3] == 0            # the limit falls exactly on rank 1's first record


def test_what_falls_back_to_one_rank(tmp_path, library, monkeypatch):
    """Lone-CR line ends (no cut point), heads longer than HEAD_CAP, and ranges with too few lines."""
    tags, text = library
    path = tmp_path / "lib.fq"
    path.write_bytes(text.replace("\n", "\r").encode("utf-8"))
    assert shard(path, 2, 500000000)[1] is None          # range 1 is empty: no '\n' after the cut
    monkeypatch.setattr(counting, "HEAD_CAP", 64)
    recs = records(text)
    giant = "".join(recs[:120]) + "@giant\n" + "A" * 200 + "\n+\n" + "#" * 200 + "\n" + "".join(recs[120:])
    path.write_bytes(giant.encode("utf-8"))
    assert shard(path, 2, 500000000)[1] is None
    monkeypatch.undo()
    assert counting.plan_trimmed_shards([5, 2, 9], [b"a\nb\nc\n", b"d\ne\n", b"f\ng\nh\n"], 10) is None
    assert counting.plan_trimmed_shards([5, 4, 9], [b"a\nb\nc\n", b"d\ne\nf\n", b"g\nh\ni\n"], 10) == [
        (0, b"d\ne\nf\n", 0, 10), (6, b"g\nh\ni\n", 2, 8), (6, b"", 3, 7)]


def test_line_ends():
    assert counting.line_ends(b"a\r\nb\rc\nd", 3) == [3, 5, 7]
    assert counting.line_ends(b"a\r\nb\r", 3) == [3, 5]
    assert counting.line_ends(b"a\r\nb\r", 3, whole=False) == [3]
    assert counting.line_ends(b"\n\n\n\n", 2) == [1, 2]
    assert counting.line_ends(b"abc", 3) == []
