"""Sharding one BGZF file across ranks, checked without a GPU: the member index of tdg_bgzf_index against
the members tests/feed_check.py writes, which files shard_files admits, and counting.plan_bgzf_share --
for 2 to 5 ranks, the owned texts of all ranks put together must be the whole text, wherever the member
cuts fall."""

import ctypes
import gzip
import os
import random

import numpy as np
import pytest

from feed_check import bgzf_block, bgzf_compress
from tagdigger_b200 import _native, counting

HEADER = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00"     # a BGZF member header, as text


def reads(n, seed=3, sep="\n"):
    rng = random.Random(seed)
    out = []
    for i in range(n):
        s = "".join(rng.choice("ACGT") for _ in range(rng.randint(30, 150)))
        out.append(sep.join(["@read%d" % i, s, "+", "I" * len(s)]) + sep)
    return "".join(out).encode("ascii")


def write_members(path, parts, level=6):
    """A file of one BGZF member per part; returns the members' offsets."""
    blocks = [bgzf_block(p, level) for p in parts]
    with open(path, "wb") as fh:
        fh.write(b"".join(blocks))
    return [int(x) for x in np.cumsum([0] + [len(b) for b in blocks[:-1]])]


# ---- tdg_bgzf_index ------------------------------------------------------------------------------

def test_index_of_stored_members_with_header_bytes_in_the_text(tmp_path):
    text = (HEADER + reads(40)) * 30
    parts = [text[i:i + 9000] for i in range(0, len(text), 9000)] + [b""]
    offs = write_members(str(tmp_path / "a.fq.gz"), parts, level=0)
    off, isize = _native.bgzf_index(str(tmp_path / "a.fq.gz"))
    assert off.tolist() == offs
    assert isize.tolist() == [len(p) for p in parts]


def test_index_with_empty_members_and_without_eof_marker(tmp_path):
    text = reads(400)
    parts = []
    for i in range(0, len(text), 7000):
        parts += [text[i:i + 7000], b""] if i % 21000 == 0 else [text[i:i + 7000]]
    path = str(tmp_path / "a.fq.gz")
    offs = write_members(path, parts)
    assert parts[-1] != b""                                   # no end-of-file marker: still a clean chain
    off, isize = _native.bgzf_index(path)
    assert off.tolist() == offs and isize.tolist() == [len(p) for p in parts]
    assert int(isize.sum()) == len(text)


@pytest.mark.parametrize("damage", ["truncated last member", "gzip member after BGZF", "first member not BGZF",
                                    "empty file"])
def test_index_refuses_a_chain_that_is_not_clean(tmp_path, damage):
    text = reads(300)
    data = bgzf_compress(text, block=10000)
    if damage == "truncated last member":
        data = bgzf_compress(text, block=10000, eof_marker=False)[:-3]
    elif damage == "gzip member after BGZF":
        data = data + gzip.compress(text)
    elif damage == "first member not BGZF":
        data = gzip.compress(text[:500]) + data
    else:
        data = b""
    path = str(tmp_path / "a.fq.gz")
    with open(path, "wb") as fh:
        fh.write(data)
    assert _native.bgzf_index(path) is None
    assert _native.lib().tdg_bgzf_index(os.fsencode(path), None, None, 0, ctypes.byref(ctypes.c_size_t())) == _native.TDG_ERR_GZIP


def test_index_asks_for_its_room(tmp_path):
    path = str(tmp_path / "a.fq.gz")
    with open(path, "wb") as fh:
        fh.write(bgzf_compress(reads(300), block=10000))
    L = _native.lib()
    n = ctypes.c_size_t(0)
    assert L.tdg_bgzf_index(os.fsencode(path), None, None, 0, ctypes.byref(n)) == _native.TDG_OK
    assert n.value == len(_native.bgzf_index(path)[0])
    off = np.zeros(n.value, dtype=np.uint64)
    isize = np.zeros(n.value, dtype=np.uint32)
    assert L.tdg_bgzf_index(os.fsencode(path), off.ctypes.data, isize.ctypes.data, n.value - 1, ctypes.byref(n)) == _native.TDG_ERR_ARG
    with pytest.raises(_native.TdgError) as e:
        _native.bgzf_index(str(tmp_path / "missing.gz"))
    assert e.value.code == _native.TDG_ERR_IO


def test_shard_files_admits_clean_bgzf_chains_only(tmp_path, monkeypatch):
    monkeypatch.setattr(counting, "SHARD_MIN_BYTES", 1024)
    monkeypatch.delenv("TDG_GZDEV", raising=False)
    text = reads(2000)
    files = {"bgzf.fq.gz": bgzf_compress(text, block=20000), "plain.fq.gz": gzip.compress(text),
             "mixed.fq.gz": bgzf_compress(text, block=20000, eof_marker=False) + gzip.compress(text), "text.fq": text}
    for name, data in files.items():
        with open(str(tmp_path / name), "wb") as fh:
            fh.write(data)
    names = [str(tmp_path / n) for n in sorted(files)]
    split = counting.shard_files(names, 5)
    assert sorted(os.path.basename(f) for f in split) == ["bgzf.fq.gz", "text.fq"]
    assert split[str(tmp_path / "text.fq")] is None
    assert int(split[str(tmp_path / "bgzf.fq.gz")][1].sum()) == len(text)
    monkeypatch.setenv("TDG_GZDEV", "0")
    assert list(counting.shard_files(names, 5)) == [str(tmp_path / "text.fq")]


# ---- plan_bgzf_share ----------------------------------------------------------------------------

def plan(parts, world, cap=None):
    """Every rank's share of a file of members ``parts`` (100 file bytes each, so the member cuts are
    c[r] = ceil(m * r / world)), or None when a rank refuses."""
    text = b"".join(parts)
    isize = np.array([len(p) for p in parts], dtype=np.uint32)
    off = np.arange(len(parts), dtype=np.uint64) * 100
    t = np.concatenate([[0], np.cumsum(isize.astype(np.int64))])
    calls = []

    def text_of(k0, k1):
        calls.append((k0, k1))
        return text[t[k0]:t[k1]]
    shares = [counting.plan_bgzf_share(off, isize, 100 * len(parts), r, world, text_of, cap) for r in range(world)]
    if any(s is None for s in shares):
        return None
    for lo, hi, k_first, k_last, front, back in shares:
        assert text[lo:t[k_first]] == front and text[t[k_last]:hi] == back and k_first <= k_last
        assert lo == 0 or text[lo - 1:lo] == b"\n"                    # every range starts at a line start
    assert b"".join(text[s[0]:s[1]] for s in shares) == text
    return shares


def split_at(text, cuts):
    cuts = sorted(set(c for c in cuts if 0 < c < len(text)))
    return [text[a:b] for a, b in zip([0] + cuts, cuts + [len(text)])]


def line_offsets(text, after=b"\n"):
    return [i + len(after) for i in range(len(text)) if text.startswith(after, i)]


@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_cuts_mid_line_and_at_line_ends(world):
    text = reads(300)
    starts = [0] + line_offsets(text)[:-1]
    assert plan(split_at(text, [s + 7 for s in starts[::3]]), world)             # every member cut mid-line
    assert plan(split_at(text, starts[::5]), world)                               # every member cut at a line end
    assert plan(split_at(text, range(0, len(text), 777)), world)


@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_cuts_between_cr_and_lf(world):
    text = reads(300, sep="\r\n")
    crs = [i + 1 for i in range(len(text)) if text[i:i + 1] == b"\r"]
    shares = plan(split_at(text, crs[::4]), world)
    assert shares
    assert all(text[s[0] - 2:s[0]] == b"\r\n" for s in shares[1:])


@pytest.mark.parametrize("line", [0, 1, 2, 3])
@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_cuts_inside_each_line_of_a_record(world, line):
    text = reads(300)
    starts = [0] + line_offsets(text)[:-1]
    assert plan(split_at(text, [s + 1 for s in starts[line::4][::2]]), world)


@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_empty_members_at_the_cuts(world):
    text = reads(300)
    parts = split_at(text, range(0, len(text), 900))
    with_empty = []
    for p in parts:
        with_empty += [p, b"", b""]
    assert plan(with_empty, world)


@pytest.mark.parametrize("world", [2, 3, 4, 5])
def test_a_line_longer_than_a_member(world):
    recs = reads(200).split(b"\n")
    giant = b"\n".join(recs[:len(recs) // 2] + [b"ACGT" * 20000] + recs[len(recs) // 2:])
    parts = split_at(giant, range(0, len(giant), 3000))
    if world == 2:
        assert b"\n" not in parts[(len(parts) + 1) // 2]        # the one cut lands inside the long line
    # within the look-ahead cap: sharded at world 2; with more ranks a range may lie wholly inside the long
    # line (no '\n' of its own: the file is counted whole), otherwise plan checks the owned texts
    shares = plan(parts, world)
    assert shares or world > 2
    if world == 2:
        assert plan(parts, world, cap=10000) is None


def test_look_ahead_cap():
    text = reads(100)
    giant = text + b"A" * 60000 + b"\n" + text
    parts = split_at(giant, range(0, len(giant), 2000))
    assert plan(parts, 2) is not None
    assert plan(parts, 2, cap=70000) is not None
    assert plan(parts, 2, cap=20000) is None
    lone_cr = text.replace(b"\n", b"\r")
    assert plan(split_at(lone_cr, range(0, len(lone_cr), 2000)), 3) is None


def test_plan_over_a_real_index(tmp_path):
    """The planner over tdg_bgzf_index of a written file, text taken from zlib."""
    text = reads(3000)
    path = str(tmp_path / "a.fq.gz")
    with open(path, "wb") as fh:
        fh.write(bgzf_compress(text, block=6000))
    off, isize = _native.bgzf_index(path)
    t = np.concatenate([[0], np.cumsum(isize.astype(np.int64))])
    for world in (2, 3, 4, 5):
        shares = [counting.plan_bgzf_share(off, isize, os.path.getsize(path), r, world, lambda a, b: text[t[a]:t[b]])
                  for r in range(world)]
        assert b"".join(text[s[0]:s[1]] for s in shares) == text
