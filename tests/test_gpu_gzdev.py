"""The device-side gzip feed (tagdigger_b200/csrc/tdg_gzdev.cuh) on a B200: the bytes it inflates
must be those Python's gzip module reads (gzip.open of /root/reference/tagdigger_fun.py:240-241),
and files counted through it must give the oracle's matrix -- whatever the block kinds, the chunk
geometry and the place where the host reader has to take over.  The same streams run through the
per-lane code on the CPU in tests/test_gzlane_cpu.py."""

import gzip
import io
import random
import struct
import zlib

import numpy as np
import pytest

from oracle import c_oracle
from tagdigger_b200 import _native, counting, synth
from test_feed_cpu import _deflate_pieces, _fastq_like

pytestmark = pytest.mark.gpu


def _inflate(tmp_path, blob, cap, name="x.gz"):
    p = str(tmp_path / name)
    with open(p, "wb") as fh:
        fh.write(blob)
    return counting.get_engine(0).gz_inflate_host(p, cap)


@pytest.mark.parametrize("level", [1, 6, 9])
@pytest.mark.parametrize("chunk,max_chunks", [(0, 0), (1 << 16, 37), (40000, 7), (4096, 3000)])
def test_device_feed_fastq(tmp_path, monkeypatch, level, chunk, max_chunks):
    if chunk:
        monkeypatch.setenv("TDG_GZDEV_CHUNK", str(chunk))
        monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", str(max_chunks))
    data = _fastq_like(10 + level, 24 << 20 if not chunk else 6 << 20)
    out, info, ms = _inflate(tmp_path, gzip.compress(data, level), len(data) + 100)
    assert out == data
    if chunk == 0 or chunk >= 1 << 16:
        assert info["mode"] == 0 and info["accepted"] >= 0.9 * info["chunks"], info


def test_device_feed_block_kinds(tmp_path, monkeypatch):
    r = random.Random(7)
    text = _fastq_like(3, 3 << 20)
    noise = r.randbytes(1 << 20)
    pieces = [
        (text[:900000], 6, zlib.Z_DEFAULT_STRATEGY, zlib.Z_FULL_FLUSH),
        (noise, 6, zlib.Z_DEFAULT_STRATEGY, zlib.Z_FULL_FLUSH),
        (text[900000:1500000], 6, zlib.Z_FIXED, zlib.Z_FULL_FLUSH),
        (b"A" * (9 << 20), 9, zlib.Z_DEFAULT_STRATEGY, zlib.Z_FULL_FLUSH),
        (text[1500000:], 1, zlib.Z_DEFAULT_STRATEGY, zlib.Z_FULL_FLUSH),
        (noise[:70000], 0, zlib.Z_DEFAULT_STRATEGY, zlib.Z_FULL_FLUSH),
        (text[:300000], 9, zlib.Z_HUFFMAN_ONLY, zlib.Z_FULL_FLUSH),
        (text[:300000], 9, zlib.Z_RLE, zlib.Z_FULL_FLUSH),
    ]
    blob, raw = _deflate_pieces(pieces)
    for chunk, max_chunks in ((1 << 16, 16), (20000, 64), (1 << 20, 4)):
        monkeypatch.setenv("TDG_GZDEV_CHUNK", str(chunk))
        monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", str(max_chunks))
        out, info, ms = _inflate(tmp_path, blob, len(raw) + 100)
        assert out == raw, (chunk, info)


def test_device_feed_each_kind_alone_and_long_codes(tmp_path, monkeypatch):
    monkeypatch.setenv("TDG_GZDEV_CHUNK", str(1 << 15))
    text = _fastq_like(4, 1 << 20)
    for strategy, level in ((zlib.Z_FIXED, 6), (zlib.Z_HUFFMAN_ONLY, 6), (zlib.Z_RLE, 6), (zlib.Z_DEFAULT_STRATEGY, 0),
                            (zlib.Z_FILTERED, 9)):
        co = zlib.compressobj(level, zlib.DEFLATED, 31, 9, strategy)
        out, info, ms = _inflate(tmp_path, co.compress(text) + co.flush(), len(text) + 100)
        assert out == text, (strategy, level, info)
    r = random.Random(11)
    vals = []
    for _ in range(2 << 20):
        v = 0
        while v < 255 and r.random() < 0.72:
            v += 1
        vals.append(v)
    data = bytes(vals)
    for level in (1, 9):
        out, info, ms = _inflate(tmp_path, gzip.compress(data, level), len(data) + 100)
        assert out == data, info


def test_device_feed_members_headers_and_tails(tmp_path, monkeypatch):
    data = _fastq_like(5, 4 << 20)
    cuts = [0, 10, 10, 70000, 70001, 900000, 2500000, len(data)]
    blob = b""
    for a, b in zip(cuts, cuts[1:]):
        bio = io.BytesIO()
        with gzip.GzipFile(filename="part%d.fq" % a, mode="wb", fileobj=bio, compresslevel=1 + a % 9, mtime=a) as g:
            g.write(data[a:b])
        blob += bio.getvalue()
    extra = b"XY\x03\x00abc"
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = co.compress(data[:5000]) + co.flush()
    blob += (b"\x1f\x8b\x08\x14\x00\x00\x00\x00\x00\xff" + struct.pack("<H", len(extra)) + extra + b"a comment\x00" + body +
             struct.pack("<II", zlib.crc32(data[:5000]), 5000))
    want = data + data[:5000]
    for chunk in (50000, 4096, 1 << 20):
        monkeypatch.setenv("TDG_GZDEV_CHUNK", str(chunk))
        out, info, ms = _inflate(tmp_path, blob, len(want) + 100)
        assert out == want, info
    for tail in (b"\0" * 1000, b"garbage that is not gzip", b"\x1f"):
        out, info, ms = _inflate(tmp_path, blob + tail, len(want) + 100)
        assert out == want, (tail[:8], info)
    # sync flush points keep the window
    text = _fastq_like(4, 2 << 20)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = b""
    for i in range(0, len(text), 50000):
        body += co.compress(text[i:i + 50000]) + co.flush(zlib.Z_SYNC_FLUSH)
    body += co.flush()
    blob = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + body + struct.pack("<II", zlib.crc32(text), len(text))
    monkeypatch.setenv("TDG_GZDEV_CHUNK", "30000")
    out, info, ms = _inflate(tmp_path, blob, len(text) + 100)
    assert out == text


def test_device_feed_damaged_streams_end_like_the_host_path(tmp_path, monkeypatch):
    """Same error (code and zlib's words) as the host feeder alone -- the device feed hands the
    stream over in front of the defect."""
    monkeypatch.setenv("TDG_GZDEV_CHUNK", "40000")
    data = _fastq_like(6, 3 << 20)
    good = gzip.compress(data, 6)
    bad = bytearray(good)
    bad[len(bad) // 2] ^= 0x10
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = co.compress(data) + co.flush()
    head = b"\x1f\x8b\x08\x02\x00\x00\x00\x00\x00\xff"
    cases = {
        "fhcrc": head + struct.pack("<H", zlib.crc32(head) & 0xFFFF) + body + struct.pack("<II", zlib.crc32(data), len(data)),
        "flipped bit": bytes(bad),
        "wrong crc": good[:-8] + struct.pack("<II", zlib.crc32(data) ^ 1, len(data)),
        "wrong isize": good[:-8] + struct.pack("<II", zlib.crc32(data), len(data) + 1),
        "truncated": good[:len(good) * 2 // 3],
        "truncated trailer": good[:-3],
        "bad second header": good + b"\x1f\x8b\x09\x00" + good[4:],
        "second member corrupt": good + bytes(bad),
        "reserved flag": good + b"\x1f\x8b\x08\x80" + good[4:],
    }
    from feed_check import FeedError, read_file
    eng = counting.get_engine(0)
    p = str(tmp_path / "odd.gz")
    for name, blob in cases.items():
        with open(p, "wb") as fh:
            fh.write(blob)
        try:
            want = read_file(p, True, 1 << 20, cap=2 * len(data) + 100)[0]          # the host feeder alone (tdg_feed.h)
        except FeedError as e:
            want = (e.code, type(counting._gzip_exception(str(e).split(": ", 1)[1])))
        try:
            got = eng.gz_inflate_host(p, 2 * len(data) + 100)[0]
        except _native.TdgError as e:
            got = (e.code, type(counting._gzip_exception(e.message)))       # the exception find_tags_fastq raises
        assert got == want, name
        if name not in ("fhcrc", "reserved flag"):
            # ... which is what the reference's gzip.open does with these files: an exception
            assert isinstance(got, tuple) and got[0] == _native.TDG_ERR_GZIP, name
            with pytest.raises(Exception):
                gzip.open(p, "rb").read()


def test_device_feed_small_symbol_buffers_hand_over(tmp_path, monkeypatch):
    monkeypatch.setenv("TDG_GZDEV_CHUNK", str(1 << 14))
    monkeypatch.setenv("TDG_GZDEV_SYMCAP", str(8 << 14))
    monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", "8")
    data = b"ACGT" * (3 << 20) + _fastq_like(2, 1 << 20)
    out, info, ms = _inflate(tmp_path, gzip.compress(data, 6), len(data) + 100)
    assert out == data and info["mode"] == 1


def test_device_feed_random_streams(tmp_path, monkeypatch):
    r = random.Random(2024)
    for case in range(10):
        parts = []
        for _ in range(r.randint(3, 30)):
            kind = r.random()
            if kind < 0.3:
                parts.append(r.randbytes(r.randint(1, 40000)))
            elif kind < 0.6:
                parts.append(bytes(r.choice(b"ACGTN\n@+I") for _ in range(r.randint(1, 60000))))
            elif kind < 0.8 and parts:
                src = parts[r.randrange(len(parts))]
                parts.append(src[:r.randint(0, len(src))] * r.randint(1, 4))
            else:
                parts.append(bytes([r.randrange(256)]) * r.randint(1, 100000))
        data = b"".join(parts)
        monkeypatch.setenv("TDG_GZDEV_CHUNK", str(r.choice((4096, 8192, 1 << 15, 1 << 16))))
        monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", str(r.randint(1, 40)))
        out, info, ms = _inflate(tmp_path, gzip.compress(data, r.choice((1, 4, 6, 9))), len(data) + 100)
        assert out == data, (case, info)


# ---------------------------------------------------------------------------------------------
# counting through the device feed

def _tables(seed=3):
    rng = np.random.default_rng(seed)
    bcs = synth.make_barcodes(24, rng)
    _, _, seqs = synth.make_marker_pairs(400, rng)
    return rng, bcs, [s for p in seqs for s in p]


@pytest.mark.parametrize("ending", ["lf", "crlf", "no final newline"])
def test_count_gzip_file_on_the_device(tmp_path, ending, capsys):
    rng, bcs, tags = _tables()
    fq, _ = synth.make_fastq(150000, bcs, tags, rng)
    if ending == "crlf":
        fq = fq.replace(b"\n", b"\r\n")
    elif ending == "no final newline":
        fq = fq[:-1]
    assert len(gzip.compress(fq, 1)) > 9 << 20
    p = str(tmp_path / "reads.fq.gz")
    with open(p, "wb") as fh:
        fh.write(gzip.compress(fq, 1))
    want, wtot = c_oracle.Counter(bcs, tags).count(fq)
    eng = counting.get_engine(0)
    before = eng.launch_count()
    tot = []
    got = np.asarray(counting.find_tags_fastq(p, bcs, tags, totals=tot))
    assert tot[:3] == wtot and (got == want).all()
    # the device feed did the inflating -- with the reference's default maxreads (5e9) in the call
    info = eng.last_file_info()
    assert info["mode"] == 0 and info["rounds"] >= 1 and eng.launch_count() > before, info


def test_count_gzip_members_and_utf8_on_the_device(tmp_path, monkeypatch):
    rng, bcs, tags = _tables(4)
    fq, _ = synth.make_fastq(120000, bcs, tags, rng)
    lines = fq.split(b"\n")
    lines[4000] = lines[4000] + " séquence ü".encode()           # valid UTF-8 in a header line
    fq = b"\n".join(lines)
    third = len(fq) // 3
    blob = gzip.compress(fq[:third], 1) + gzip.compress(fq[third:2 * third], 6) + gzip.compress(fq[2 * third:], 1)
    p = str(tmp_path / "members.fq.gz")
    with open(p, "wb") as fh:
        fh.write(blob)
    want, wtot = c_oracle.Counter(bcs, tags).count(fq)
    tot = []
    got = np.asarray(counting.find_tags_fastq(p, bcs, tags, totals=tot))
    assert tot[:3] == wtot and (got == want).all()
    # invalid UTF-8 far into the file: the reference's text-mode read raises
    lines[300000] = lines[300000][:5] + b"\xff" + lines[300000][5:]
    with open(p, "wb") as fh:
        fh.write(gzip.compress(b"\n".join(lines), 1))
    with pytest.raises(UnicodeDecodeError):
        counting.find_tags_fastq(p, bcs, tags)
    # a damaged stream: counts never come back, the reference's exception does
    bad = bytearray(gzip.compress(fq, 1))
    bad[len(bad) * 3 // 4] ^= 0x20
    with open(p, "wb") as fh:
        fh.write(bytes(bad))
    with pytest.raises((zlib.error, gzip.BadGzipFile, EOFError)):
        counting.find_tags_fastq(p, bcs, tags)
    # and the same file with the device feed switched off gives the same matrix as with it
    with open(p, "wb") as fh:
        fh.write(blob)
    monkeypatch.setenv("TDG_GZDEV", "0")
    host = np.asarray(counting.find_tags_fastq(p, bcs, tags))
    assert (host == want).all()


def test_release_scratch_and_inflate_again(tmp_path):
    """tdg_release_scratch gives the feed's working buffers back; the next file allocates them again."""
    data = _fastq_like(12, 6 << 20)
    eng = counting.get_engine(0)
    out, info, ms = _inflate(tmp_path, gzip.compress(data, 6), len(data) + 100)
    assert out == data
    eng.release_scratch()
    out, info, ms = _inflate(tmp_path, gzip.compress(data, 1), len(data) + 100)
    assert out == data and info["mode"] == 0


def test_device_memory_shortage_hands_over_to_the_host(tmp_path, monkeypatch):
    """A buffer that cannot be had (simulated) is not the file's fault: the host reader finishes it,
    from the state the round began in -- inside a gzip stream or at a BGZF member."""
    from feed_check import bgzf_compress
    data = _fastq_like(13, 8 << 20)
    monkeypatch.setenv("TDG_GZDEV_CHUNK", "65536")
    for blob, max_chunks in ((gzip.compress(data, 6), 16),
                             (bgzf_compress(data), 20)):                   # about 130 members: several rounds
        monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", str(max_chunks))
        for at in (0, 2):
            monkeypatch.setenv("TDG_GZDEV_OOM_ROUND", str(at))
            out, info, ms = _inflate(tmp_path, blob, len(data) + 100)
            assert out == data and info["mode"] == 1 and info["rounds"] == at, (max_chunks, at, info)


@pytest.mark.parametrize("max_chunks", [37, 5])
def test_count_gzip_file_in_many_rounds(tmp_path, monkeypatch, max_chunks):
    """Rounds of a few chunks: the next round's bytes are prefetched, lines are carried from round to round."""
    monkeypatch.setenv("TDG_GZDEV_CHUNK", "65536")
    monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", str(max_chunks))
    rng, bcs, tags = _tables(5)
    fq, _ = synth.make_fastq(150000, bcs, tags, rng)
    p = str(tmp_path / "reads.fq.gz")
    with open(p, "wb") as fh:
        fh.write(gzip.compress(fq, 1))
    want, wtot = c_oracle.Counter(bcs, tags).count(fq)
    tot = []
    got = np.asarray(counting.find_tags_fastq(p, bcs, tags, totals=tot))
    assert tot[:3] == wtot and (got == want).all()
    info = counting.get_engine(0).gz_inflate_host(p, len(fq) + 100)[1]
    assert info["mode"] == 0 and info["rounds"] > 3


# ---------------------------------------------------------------------------------------------
# BGZF: every member is its own stream -- one lane per member, nothing speculative

def test_device_feed_bgzf(tmp_path, monkeypatch):
    from feed_check import bgzf_block, bgzf_compress
    data = _fastq_like(14, 12 << 20)
    eng = counting.get_engine(0)
    for blob, want in ((bgzf_compress(data), data),
                       (bgzf_compress(data[:3000000], block=777, eof_marker=False), data[:3000000]),      # tiny members, no EOF marker
                       (bgzf_compress(data[:1 << 20], level=1) + bgzf_compress(data[1 << 20:5 << 20], level=9), data[:5 << 20])):
        out, info, ms = _inflate(tmp_path, blob, len(want) + 100, name="b.gz")
        assert out == want and info["mode"] == 0 and info["accepted"] == info["chunks"] > 0, info
    # few lanes per round
    monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", "13")
    out, info, ms = _inflate(tmp_path, bgzf_compress(data[:4 << 20]), (4 << 20) + 100, name="b.gz")
    assert out == data[:4 << 20] and info["rounds"] > 4
    monkeypatch.delenv("TDG_GZDEV_MAXCHUNKS")
    # BGZF members followed by an ordinary member: the host feeder continues there
    half = 3 << 20
    blob = bgzf_compress(data[:half], eof_marker=False) + gzip.compress(data[half:2 * half])
    out, info, ms = _inflate(tmp_path, blob, 2 * half + 100, name="b.gz")
    assert out == data[:2 * half] and info["mode"] == 1
    # a damaged member, a wrong CRC, a wrong length: a gzip error, as from the host feeder
    good = bgzf_compress(data[:2 << 20])
    for kind in ("flip", "crc", "isize"):
        bad = bytearray(good)
        first = struct.unpack("<H", good[16:18])[0] + 1                  # size of the first member
        if kind == "flip":
            bad[len(bad) // 2] ^= 0x55
        elif kind == "crc":
            bad[first - 8] ^= 1
        else:
            bad[first - 4] ^= 1
        p = str(tmp_path / "bad.gz")
        with open(p, "wb") as fh:
            fh.write(bytes(bad))
        with pytest.raises(_native.TdgError) as e:
            eng.gz_inflate_host(p, (2 << 20) + 100)
        assert e.value.code == _native.TDG_ERR_GZIP, kind
        with pytest.raises(Exception):
            gzip.open(p, "rb").read()


def test_count_bgzf_file_on_the_device(tmp_path, monkeypatch):
    from feed_check import bgzf_compress
    monkeypatch.setenv("TDG_GZDEV_MIN", "0")
    rng, bcs, tags = _tables(6)
    fq, _ = synth.make_fastq(60000, bcs, tags, rng)
    fq = fq[:-1]                                                         # no final newline
    p = str(tmp_path / "reads.fq.gz")
    with open(p, "wb") as fh:
        fh.write(bgzf_compress(fq))
    want, wtot = c_oracle.Counter(bcs, tags).count(fq)
    eng = counting.get_engine(0)
    before = eng.launch_count()
    tot = []
    got = np.asarray(counting.find_tags_fastq(p, bcs, tags, totals=tot))
    assert tot[:3] == wtot and (got == want).all()
    assert eng.gz_inflate_host(p, len(fq) + 100)[1]["mode"] == 0 and eng.launch_count() > before


def test_count_files_reads_the_next_file_ahead(tmp_path):
    """count_files names every file's successor to the library (tdg_count_file2): plain files, small gzip files,
    an empty file and a file without a final newline in one key give the per-file oracle rows; a file that is
    missing raises when its turn comes, not before."""
    rng, bcs, tags = _tables(8)
    bckeys, want_rows, names = {}, [], []
    for i in range(9):
        fq, _ = synth.make_fastq(4000 + 700 * i, bcs[:4], tags, rng)
        if i == 3:
            fq = b""
        if i == 5:
            fq = fq[:-1]
        name = str(tmp_path / ("s%02d.fq%s" % (i, ".gz" if i % 3 == 1 else "")))
        with open(name, "wb") as fh:
            fh.write(gzip.compress(fq) if name.endswith("gz") else fq)
        bckeys[name] = [list(bcs[:4]), ["S%d_%d" % (i, b) for b in range(4)]]
        want_rows.append(c_oracle.Counter(bcs[:4], tags).count(fq)[0])
        names.append(name)
    samples, counts = counting.count_files(bckeys, tags, as_array=True)
    assert len(samples) == 36 and (np.asarray(counts) == np.concatenate(want_rows)).all()
    # twice in a row (the reader started for a file that never came is dropped), then with a hole in the key
    samples, counts = counting.count_files(bckeys, tags, as_array=True)
    assert (np.asarray(counts) == np.concatenate(want_rows)).all()
    import os
    os.remove(names[4])
    with pytest.raises(FileNotFoundError):
        counting.count_files(bckeys, tags)
    got = np.asarray(counting.find_tags_fastq(names[5], bcs[:4], tags))
    assert (got == want_rows[5]).all()


# ---------------------------------------------------------------------------------------------
# the read limit (maxreads, default 5e9) on the host side of tdg_count_file

def _with_engine(chunk_bytes):
    """A process-wide engine with small pieces, so that megabytes behave like the tens of gigabytes the default
    limit is about; returns a function that puts the old engine back."""
    old = counting._engines.pop(0, None)
    counting._engines[0] = _native.Engine(0, chunk_bytes=chunk_bytes)

    def restore():
        counting._engines.pop(0).close()
        if old is not None:
            counting._engines[0] = old
    return restore


@pytest.mark.parametrize("kind", ["plain", "gzip", "gzip on the device", "gzip on the device, tiny rounds", "bgzf on the device", "crlf"])
def test_read_limit_is_looked_for_only_where_it_can_be(tmp_path, monkeypatch, kind):
    """Limits far beyond the file cost nothing (no pass over the bytes on the host, device gzip feed in use); limits
    inside the file stop the reader exactly there -- a defect behind the limit is never met; counts equal the
    oracle's for every limit."""
    from feed_check import bgzf_compress
    rng, bcs, tags = _tables(9)
    fq, _ = synth.make_fastq(30000, bcs, tags, rng)
    if kind == "crlf":
        fq = fq.replace(b"\n", b"\r\n")
    nreads = 30000
    bad_tail = b"@x\nAC\xffGT\n+\nIIII\n"                      # invalid UTF-8: the reference would raise if it got there
    p = str(tmp_path / ("r.fq" + ("" if kind in ("plain", "crlf") else ".gz")))
    restore = _with_engine(1 << 16)
    try:
        if "device" in kind:
            monkeypatch.setenv("TDG_GZDEV_MIN", "0")
            monkeypatch.setenv("TDG_GZDEV_CHUNK", "16384" if "tiny" in kind else "32768")
            monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", "2" if "tiny" in kind else "40")
        else:
            monkeypatch.setenv("TDG_GZDEV", "0")
        for limit in (5e9, 20000, 29999, 30000, 30001, 16500, 123):
            damaged = limit <= nreads
            data = fq + (bad_tail if damaged else b"")
            with open(p, "wb") as fh:
                if kind in ("plain", "crlf"):
                    fh.write(data)
                elif kind.startswith("bgzf"):
                    fh.write(bgzf_compress(data, block=4000))
                else:
                    fh.write(gzip.compress(data, 1))
            want, wtot = c_oracle.Counter(bcs, tags).count(fq, limit)[:2]
            tot = []
            got = np.asarray(counting.find_tags_fastq(p, bcs, tags, maxreads=limit, totals=tot))
            assert tot[:3] == wtot and (got == want).all(), (kind, limit)
            info = counting.get_engine(0).last_file_info()
            if "device" in kind and limit == 5e9:
                assert info["mode"] == 0 and info["rounds"] >= 1, (kind, info)         # the default limit keeps nothing from the device
            if "tiny" in kind and limit == 20000:
                # rounds of 65 KB of text fit under the limit's line for a while: the device feeds them, then the host
                # feeder takes over and stops at the limit
                assert info["mode"] == 1 and info["rounds"] >= 10, info
        # ... and without a limit in the way the damaged tail IS met
        with pytest.raises(UnicodeDecodeError):
            counting.find_tags_fastq(p, bcs, tags, maxreads=nreads + 2)
    finally:
        restore()
