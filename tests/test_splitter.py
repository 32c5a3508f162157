"""Barcode splitter (SURVEY.md 8(f) rank 2, rows A8 + barcodeSplitter): output files of
tagdigger_b200.splitter.barcodeSplitter against the files recorded from the reference
(tests/golden/splitter.json) and against the oracle's record-by-record restatement on
fresh inputs; the decisions come from the GPU (tdg_split_batch)."""

import base64
import contextlib
import gzip
import io
import os
import random

import pytest

from conftest import NO_REFERENCE, have_reference, import_reference, load_golden, materialize
from helpers import rand_seq
from oracle import tagdigger_oracle as orc
from tagdigger_b200 import barcode_splitter_script, hostio

GOLD = load_golden("splitter.json")


def test_cli_surface():
    p = barcode_splitter_script.build_parser()
    flags = set()
    for a in p._actions:
        flags.update(a.option_strings)
    assert {"-b", "--barcodefile", "-a", "--adapter"} <= flags
    with pytest.raises(SystemExit):
        p.parse_args(["-b", "k.csv", "-a", "NoSuch-Adapter"])
    assert sorted(hostio.adapters) == ["NsiI-MspI-Clark", "NsiI-MspI-Hall", "PstI-MspI-Clark", "PstI-MspI-Hall",
                                       "PstI-MspI-Poland"]


def _oracle_files(text_lines, barcodes, cutsite, adapter, maxreads=500000000):
    bufs = [io.StringIO() for _ in barcodes]
    with contextlib.redirect_stdout(io.StringIO()):
        for b, lines, _ in orc.split_records(text_lines, barcodes, cutsite, adapter, maxreads):
            bufs[b].write("".join(ln + "\n" for ln in lines))
    return [b.getvalue().encode() for b in bufs]


def _make_input(rng, barcodes, cutsite, adapter, n, newline="\n"):
    full0 = adapter[0][0].replace("^", "")
    full1 = adapter[1][0].replace("^", "")
    a0 = adapter[0][0][:adapter[0][0].find("^")] + adapter[0][1]
    out = []
    for i in range(n):
        bc = rng.choice(barcodes)
        a1 = adapter[1][0][:adapter[1][0].find("^")] + adapter[1][1].replace("[barcode]", hostio.reverseComplement(bc))
        k = rng.random()
        insert = rand_seq(rng, rng.randint(0, 110))
        if k < 0.3:
            tail = rng.choice([a0, a1])[:rng.randint(1, 70)]
        elif k < 0.45:
            tail = rng.choice([full0, full1]) + rand_seq(rng, rng.randint(0, 30))
        elif k < 0.55:
            tail = rng.choice([a0, a1]) + rand_seq(rng, rng.randint(1, 5))
        else:
            tail = rand_seq(rng, rng.randint(0, 30))
        head = bc + cutsite if rng.random() < 0.85 else rand_seq(rng, rng.randint(0, 12))
        s = (head + insert + tail)[:rng.choice([40, 100, 100, 150])]
        w = rng.random()
        if s and w < 0.06:
            j = rng.randrange(len(s))
            s = s[:j] + "N" + s[j + 1:]
        elif w < 0.12:
            s = s.lower()
        elif w < 0.15:
            s = "  " + s + "\t"
        q = "".join(rng.choice("ABCDEFGHIJ#@+") for _ in range(len(s.strip()) if rng.random() < 0.9 else rng.randint(0, 60)))
        c1 = "@r%d %s" % (i, rng.choice(["1:N:0", "x y", "café", ""]))
        c2 = "+" if rng.random() < 0.8 else "+" + c1[1:]
        out.append(c1 + newline + s + newline + c2 + newline + q + newline)
    return "".join(out)


@pytest.mark.gpu
def test_splitter_golden(in_tmp):
    from tagdigger_b200 import splitter
    for case in GOLD:
        materialize(case["files"], in_tmp)
        inp, barcodes, outs = case["args"]
        kw = dict(case["kwargs"])
        kw["adapter"] = [tuple(x) for x in kw["adapter"]]
        with contextlib.redirect_stdout(io.StringIO()):
            assert splitter.barcodeSplitter(inp, barcodes, outs, **kw) is None
        for name in outs:
            with open(name, "rb") as fh:
                assert fh.read() == base64.b64decode(case["outfiles"][name]), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(hostio.adapters))
def test_splitter_against_oracle(name, in_tmp, monkeypatch):
    from tagdigger_b200 import splitter
    monkeypatch.setattr(splitter, "BLOCK_READS", 700)          # several GPU blocks per file
    rng = random.Random(len(name) * 7 + 1)
    adapter = hostio.adapters[name]
    cutsite = "TGCAG" if name.startswith("PstI") else "TGCAT"
    barcodes = []
    while len(barcodes) < 9:
        b = rand_seq(rng, rng.randint(4, 9))
        pat = b + cutsite
        if not any(p.startswith(pat) or pat.startswith(p) for p in (x + cutsite for x in barcodes)):
            barcodes.append(b)
    for newline, gz, maxreads in (("\n", False, 500000000), ("\r\n", True, 1234), ("\n", False, 1)):
        text = _make_input(rng, barcodes, cutsite, adapter, 3000, newline)
        inp = "in.fq.gz" if gz else "in.fq"
        data = text.encode("utf-8")
        with open(inp, "wb") as fh:
            fh.write(gzip.compress(data) if gz else data)
        outs = ["o%d.fq" % i for i in range(len(barcodes))]
        with contextlib.redirect_stdout(io.StringIO()):
            splitter.barcodeSplitter(inp, barcodes, outs, cutsite=cutsite, adapter=adapter, maxreads=maxreads)
        want = _oracle_files(io.StringIO(text, newline=None), barcodes, cutsite, adapter, maxreads)
        for o, w in zip(outs, want):
            with open(o, "rb") as fh:
                assert fh.read() == w, (name, newline, o)
    splitter.writeMD5sums(outs[:2], "md5.csv")
    assert open("md5.csv").read().splitlines()[0] == "File name,MD5 sum"


def _check_against_oracle(splitter, text, barcodes, cutsite, adapter, maxreads=500000000, gz=False, label=""):
    inp = "in.fq.gz" if gz else "in.fq"
    data = text.encode("utf-8")
    with open(inp, "wb") as fh:
        fh.write(gzip.compress(data) if gz else data)
    outs = ["o%d.fq" % i for i in range(len(barcodes))]
    got_out, want_out = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(got_out):
        splitter.barcodeSplitter(inp, barcodes, outs, cutsite=cutsite, adapter=adapter, maxreads=maxreads)
    bufs = [io.StringIO() for _ in barcodes]
    with contextlib.redirect_stdout(want_out):
        for b, lines, _ in orc.split_records(io.StringIO(text, newline=None), barcodes, cutsite, adapter, maxreads):
            bufs[b].write("".join(ln + "\n" for ln in lines))
    for o, w in zip(outs, bufs):
        with open(o, "rb") as fh:
            assert fh.read() == w.getvalue().encode(), (label, o)
    return got_out.getvalue()


@pytest.mark.gpu
@pytest.mark.parametrize("block_bytes", [1500, 40000, 64 << 20])
def test_streaming_splitter_blocks_and_text_shapes(in_tmp, monkeypatch, block_bytes):
    """The device path block by block: carries across block edges, every newline convention,
    Unicode whitespace around lines, blank lines that shift the record phase, a last line
    without terminator, a trailing partial record -- and blocks with non-ASCII sequence or
    quality lines, which take the host path in the middle of the stream."""
    from tagdigger_b200 import splitter
    monkeypatch.setattr(splitter, "BLOCK_BYTES", block_bytes)
    monkeypatch.setattr(splitter, "BLOCK_READS", 300)
    rng = random.Random(block_bytes)
    adapter = hostio.adapters["PstI-MspI-Hall"]
    barcodes = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA"]
    base = _make_input(rng, barcodes, "TGCAG", adapter, 1200)
    recs = base.split("\n")
    recs = ["\n".join(recs[i:i + 4]) + "\n" for i in range(0, len(recs) - 1, 4)]
    # Unicode whitespace around every kind of line
    for i in range(0, len(recs), 7):
        c1, s, c2, q = recs[i].split("\n")[:4]
        pad = rng.choice(["\u00a0", "\u2003", "\x85", "\u3000 ", "\x1c\x0b", " \u2028"])
        recs[i] = "\n".join([c1 + pad, pad + s + pad, c2 + pad if rng.random() < .5 else c2, q + pad + " "]) + "\n"
    ascii_text = "".join(recs)
    for name, text in (("lf", ascii_text), ("crlf", ascii_text.replace("\n", "\r\n")), ("cr", ascii_text.replace("\n", "\r")),
                       ("no final newline", ascii_text[:-1]), ("partial record", ascii_text + "@x\nACGTATGCAGTT\n"),
                       ("blank line shifts the phase", "".join(recs[:50]) + "\n" + "".join(recs[50:])),
                       ("cr at the very end", ascii_text[:-1] + "\r"), ("empty", ""), ("one newline", "\n")):
        _check_against_oracle(splitter, text, barcodes, "TGCAG", adapter, label=name)
    _check_against_oracle(splitter, ascii_text, barcodes, "TGCAG", adapter, maxreads=777, label="maxreads")
    _check_against_oracle(splitter, ascii_text.replace("\n", "\r\n"), barcodes, "TGCAG", adapter, gz=True, label="gz")
    # non-ASCII inside sequence and quality lines: those blocks go to the host
    for i in range(100, len(recs), 211):
        c1, s, c2, q = recs[i].split("\n")[:4]
        k = rng.randrange(4)
        if k == 0:
            s = s[:12] + "\u00e9" + s[12:]
        elif k == 1:
            q = "\u00df" + q
        elif k == 2:
            s = s + "\u00f1\u00f1"
            q = q + "\u4e2d"
        else:
            s = "\u00e9" + s
        recs[i] = "\n".join([c1, s, c2, q]) + "\n"
    mixed = "".join(recs)
    out = _check_against_oracle(splitter, mixed, barcodes, "TGCAG", adapter, label="non-ascii")
    assert out.count("Reads: ") == 0                       # 1,200 reads: no progress line yet
    _check_against_oracle(splitter, mixed, barcodes, "TGCAG", adapter, maxreads=450, label="non-ascii maxreads")


@pytest.mark.gpu
def test_streaming_splitter_progress_lines(in_tmp, monkeypatch):
    """The 'Reads: ...' lines every 50,000 reads carry the running counts of the reference."""
    from tagdigger_b200 import splitter
    monkeypatch.setattr(splitter, "BLOCK_BYTES", 3 << 20)
    rng = random.Random(77)
    adapter = hostio.adapters["PstI-MspI-Clark"]
    barcodes = ["ACGTA", "TTGCAC", "GGAT"]
    text = _make_input(rng, barcodes, "TGCAG", adapter, 4000) * 30           # 120,000 reads
    inp = "in.fq"
    open(inp, "w").write(text)
    outs = ["o%d.fq" % i for i in range(3)]
    got = io.StringIO()
    with contextlib.redirect_stdout(got):
        splitter.barcodeSplitter(inp, barcodes, outs, adapter=adapter)
    lines = [ln for ln in got.getvalue().splitlines() if ln.startswith("Reads: ")]
    want = []
    n = bar = clip = 0
    with contextlib.redirect_stdout(io.StringIO()):
        recs = list(orc.split_records(io.StringIO(text, newline=None), barcodes, "TGCAG", adapter, 500000000, every=True))
    for b, _, s2 in recs:
        n += 1
        bar += b > -1
        clip += b > -1 and s2 != 999
        if n % 50000 == 0:
            want.append("Reads: {0} With barcode and cut site: {1} Clipped on 3' end: {2}".format(n, bar, clip))
    assert lines == want and len(want) == 2


@pytest.mark.gpu
@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
def test_splitter_stdout_matches_reference(in_tmp):
    from tagdigger_b200 import splitter
    ref = import_reference()
    rng = random.Random(9)
    adapter = hostio.adapters["PstI-MspI-Poland"]
    barcodes = ["ACGTA", "TTGCA", "GGATC"]
    text = _make_input(rng, barcodes, "TGCAG", adapter, 500)
    open("in.fq", "w").write(text)
    got, want = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(got):
        splitter.barcodeSplitter("in.fq", barcodes, ["a0", "a1", "a2"], adapter=adapter)
    with contextlib.redirect_stdout(want):
        ref.barcodeSplitter("in.fq", barcodes, ["b0", "b1", "b2"], adapter=ref.adapters["PstI-MspI-Poland"])
    assert got.getvalue() == want.getvalue()
    for a, b in zip(["a0", "a1", "a2"], ["b0", "b1", "b2"]):
        assert open(a, "rb").read() == open(b, "rb").read()
