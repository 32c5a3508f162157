"""The splitter's BGZF encoder (csrc/tdg_bgzf.cuh) on the CPU, through the harness that runs the
kernel's phases thread by thread (tests/native/bgzf_check.cpp): Huffman code lengths, blocks built
from chosen token lists, whole members, and the compression ratio against zlib level 1."""

import contextlib
import gzip
import io
import os
import random
import sys
import zlib

import numpy as np
import pytest

import bgzf_check
from bgzf_parse import BLOCK, EOF_MEMBER, block_header, check_file, members

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check_lengths(freq, ln, maxbits):
    used = [i for i, f in enumerate(freq) if f]
    assert len(used) >= 2
    assert all(ln[i] for i in used) and not any(ln[i] for i in range(len(freq)) if not freq[i])
    assert max(ln) <= maxbits
    assert sum(2.0 ** -int(x) for x in ln if x) == 1.0              # complete: never over-subscribed or incomplete


def _fib(n):
    a, b, out = 1, 1, []
    for _ in range(n):
        out.append(a)
        a, b = b, a + b
    return out


@pytest.mark.parametrize("n,maxbits", [(286, 15), (30, 15), (19, 7)])
def test_code_lengths_fibonacci(n, maxbits):
    """Fibonacci frequencies make the unlimited Huffman code as deep as the alphabet is long."""
    k = min(n, 40)
    freq = np.zeros(n, dtype=np.uint32)
    freq[:k] = _fib(k)
    ln, f = bgzf_check.huff_lengths(freq, maxbits)
    assert max(ln) == maxbits                                     # the limit was needed and used
    _check_lengths(f, ln, maxbits)
    # the most frequent symbols keep the shortest codes
    assert all(ln[i] >= ln[i + 1] for i in range(k - 1))


@pytest.mark.parametrize("used", [[], [0], [7], [256], [0, 1], [5, 200], [284, 285]])
def test_code_lengths_few_symbols(used):
    freq = np.zeros(286, dtype=np.uint32)
    for s in used:
        freq[s] = 1000
    ln, f = bgzf_check.huff_lengths(freq, 15)
    _check_lengths(f, ln, 15)
    assert all(f[s] == 1000 for s in used)
    if len(used) < 2:                                             # zlib's rule: an unused low symbol joins
        assert sum(1 for x in f if x) == 2 and max(ln) == 1


def test_code_lengths_all_symbols():
    rng = np.random.default_rng(3)
    for trial in range(20):
        freq = rng.integers(1, 1 << rng.integers(1, 16), size=286).astype(np.uint32)
        ln, f = bgzf_check.huff_lengths(freq, 15)
        _check_lengths(f, ln, 15)
        assert (f == freq).all()


def _tokens_to_text(tokens, rng):
    """tokens: ("lit", n) or (length, distance); returns the text and its per-position match array."""
    out = bytearray()
    m = []
    for t in tokens:
        if t[0] == "lit":
            out += bytes(rng.getrandbits(8) for _ in range(t[1]))
            m += [0] * t[1]
        else:
            ln, d = t
            assert d <= len(out)
            m += [ln << 16 | (d - 1)] + [0] * (ln - 1)
            for _ in range(ln):                                   # byte by byte: overlapping copies
                out.append(out[-d])
    return bytes(out), np.asarray(m, dtype=np.uint32)


@pytest.mark.parametrize("name,tokens", [
    ("overlapping", [("lit", 1), (258, 1), (100, 1), ("lit", 3), (200, 3), (3, 2), ("lit", 20), (257, 7)]),
    ("every length", [("lit", 300)] + [(ln, 1 + (ln * 37) % 290) for ln in range(3, 259)]),
    ("every distance code", [("lit", 33000)] + [(4 + k % 250, d) for k, d in
                                                 enumerate([1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257,
                                                            385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193,
                                                            12289, 16385, 24577, 32768])]),
    ("distance 32768", [("lit", 32768), (258, 32768), (258, 32768), ("lit", 5), (3, 32768)]),
    ("one literal", [("lit", 1)]),
])
def test_block_from_tokens(name, tokens):
    rng = random.Random(len(name))
    text, m = _tokens_to_text(tokens, rng)
    assert len(text) <= BLOCK
    blob, dynamic = bgzf_check.member(text, m)
    (mem, got), = members(blob)
    assert got == text and gzip.decompress(blob) == text
    if dynamic:
        assert block_header(mem[18:-8])[0] == 2


def test_stored_fallback():
    rng = random.Random(1)
    for n in (1, 2, 1000, BLOCK - 1, BLOCK):
        data = bytes(rng.getrandbits(8) for _ in range(n))
        blob, dynamic = bgzf_check.member(data)
        assert not dynamic and len(blob) == n + 5 + 26 and gzip.decompress(blob) == data
        assert block_header(blob[18:-8])[0] == 0


def test_eof_member():
    assert bgzf_check.member(b"")[0] == EOF_MEMBER
    assert gzip.decompress(EOF_MEMBER) == b""


def _inputs():
    rng = random.Random(11)
    yield "1 byte", b"A"
    yield "all byte values", bytes(range(256)) * 3
    yield "65279", bytes(rng.choice(b"ACGT\n") for _ in range(65279))
    yield "65280", bytes(rng.choice(b"ACGT\n") for _ in range(65280))
    yield "65281", bytes(rng.choice(b"ACGT\n") for _ in range(65281))
    unit = bytes(rng.getrandbits(8) for _ in range(32768))
    yield "period 32768", (unit * 4)[:100000]
    unit = bytes(rng.getrandbits(8) for _ in range(32769))
    yield "period 32769", (unit * 4)[:100000]
    yield "skewed", bytes(rng.choices(b"eeeeeeeeeeeettttaaoinshr ", k=150000))
    yield "text", open(os.path.join(REPO, "DESIGN.md"), "rb").read()[:200000]


@pytest.mark.parametrize("name,data", list(_inputs()), ids=lambda x: x if isinstance(x, str) else "")
def test_files(name, data):
    blob = bgzf_check.compress(data)
    assert gzip.decompress(blob) == data
    ms = check_file(blob, data)
    for mem, _ in ms[:-1]:
        if mem[18] & 6 == 4:                                      # BTYPE 10
            block_header(mem[18:-8])


def test_ratio_against_zlib_level1():
    """Config-5-shaped split output (96 barcodes, adapter read-through, random qualities): the BGZF
    files are at most 5 % larger than zlib level 1 over the same 65,280-byte cuts."""
    sys.path.insert(0, os.path.join(REPO, "scripts"))
    import config5_flow
    from oracle import tagdigger_oracle as orc
    from tagdigger_b200 import hostio, synth
    rng = random.Random(5)
    nrng = np.random.default_rng(5)
    adapter = hostio.adapters["PstI-MspI-Hall"]
    barcodes = synth.make_barcodes(96, nrng)
    _, _, seqs = synth.make_marker_pairs(2000, nrng)
    tags = [s for p in seqs for s in p]
    text = config5_flow.make_reads(rng, barcodes, tags, adapter, 30000)
    bufs = [io.StringIO() for _ in barcodes]
    with contextlib.redirect_stdout(io.StringIO()):
        for b, lines, _ in orc.split_records(io.StringIO(text, newline=None), barcodes, "TGCAG", adapter, 500000000):
            bufs[b].write("".join(ln + "\n" for ln in lines))
    plain = ours = z1 = 0
    for buf in bufs:
        d = buf.getvalue().encode()
        plain += len(d)
        ours += len(bgzf_check.compress(d))
        for k in range(0, len(d), BLOCK):
            c = zlib.compressobj(1, zlib.DEFLATED, -15)
            z1 += len(c.compress(d[k:k + BLOCK]) + c.flush()) + 26
        z1 += len(EOF_MEMBER)
    assert plain > 6_000_000
    assert ours <= 1.05 * z1, (ours / plain, z1 / plain)
