"""BGZF output of the barcode splitter on the GPU (csrc/tdg_bgzf.cuh): the encoder through the Engine
calls, the splitter with bgzf=True against its own plain output, and the files read back by the
counter (device BGZF feed and host feed)."""

import base64
import contextlib
import gzip
import io
import os
import random

import numpy as np
import pytest

import bgzf_check
from bgzf_parse import BLOCK, EOF_MEMBER, check_file
from conftest import load_golden, materialize
from test_splitter import _make_input
from tagdigger_b200 import barcode_splitter_script, hostio

pytestmark = pytest.mark.gpu

ADAPTER = hostio.adapters["PstI-MspI-Hall"]


def _engine(nbar):
    """An engine with a splitter set up for nbar barcodes and BGZF output on."""
    from tagdigger_b200 import counting, matchset, trimming
    barcodes = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA"][:nbar]
    eng = counting.get_engine(0)
    barcut = hostio.combine_barcode_and_cutsite(barcodes, "TGCAG")
    patterns = matchset.effective_set(barcut, len(barcut))
    with contextlib.redirect_stdout(io.StringIO()):
        tables = trimming.trim_tables(ADAPTER, barcodes)
    eng.begin_file(patterns.patterns, patterns.index, [len(p) for p in patterns.patterns], any_base=patterns.any_base)
    eng.set_trim(tables[0], tables[1], tables[2], tables[3], tables[4])
    eng.split_begin(barcodes, 5)
    eng.split_bgzf(True)
    return eng


def _encode(eng, streams, rng):
    """Every stream appended in random pieces (the streams' calls interleaved), then finished."""
    nbar = len(streams)
    eng.split_bgzf(True)
    out = [bytearray() for _ in range(nbar)]
    pos = [0] * nbar
    while any(p < len(s) for p, s in zip(pos, streams)):
        parts = []
        for b in range(nbar):
            step = rng.choice([0, 1, 17, 4096, 65279, 65280, 65281, 200000, 3 << 20])
            parts.append(streams[b][pos[b]:pos[b] + step])
            pos[b] += len(parts[-1])
        for b, piece in enumerate(eng.bgzf_append(parts)):
            out[b] += bytes(piece)
    for b, piece in enumerate(eng.bgzf_finish()):
        out[b] += bytes(piece)
    return [bytes(o) for o in out]


def _gpu_inputs():
    rng = random.Random(21)
    from tagdigger_b200 import synth
    nrng = np.random.default_rng(2)
    bcs = synth.make_barcodes(4, nrng)
    _, _, seqs = synth.make_marker_pairs(50, nrng)
    fq, _ = synth.make_fastq(20000, bcs, [s for p in seqs for s in p], nrng)
    unit32k = bytes(rng.getrandbits(8) for _ in range(32768))
    unit32k1 = bytes(rng.getrandbits(8) for _ in range(32769))
    return [
        ("empty", b""), ("1 byte", b"x"),
        ("65279", fq[:65279]), ("65280", fq[:65280]), ("65281", fq[:65281]),
        ("10 MB of one byte", b"A" * 10_000_000),
        ("10 MB random", np.random.default_rng(5).integers(0, 256, 10_000_000, dtype=np.uint8).tobytes()),
        ("all byte values", bytes(range(256)) * 1000),
        ("period 32768", (unit32k * 8)[:250000]), ("period 32769", (unit32k1 * 8)[:250000]),
        ("skewed", bytes(rng.choices(b"eeeeeeeeeeeettttaaoinshr \n", k=400000))),
        ("fastq", fq),
    ]


@pytest.mark.parametrize("name,data", _gpu_inputs(), ids=lambda x: x if isinstance(x, str) else "")
def test_encoder_streams(name, data):
    eng = _engine(1)
    rng = random.Random(len(name))
    first, = _encode(eng, [data], rng)
    assert gzip.decompress(first) == data
    ms = check_file(first, data)
    if not data:
        assert first == EOF_MEMBER
    # other cut points, the same bytes
    second, = _encode(eng, [data], random.Random(len(name) + 99))
    assert second == first
    # the device writes what the phases write on the CPU (first members and the last one)
    for k in sorted({0, 1, 2, len(ms) - 2} & set(range(len(ms) - 1))):
        assert bgzf_check.member(ms[k][1])[0] == ms[k][0], "member %d" % k


def test_encoder_several_barcodes():
    from tagdigger_b200 import synth
    nrng = np.random.default_rng(8)
    bcs = synth.make_barcodes(4, nrng)
    _, _, seqs = synth.make_marker_pairs(50, nrng)
    streams = [synth.make_fastq(n, bcs, [s for p in seqs for s in p], nrng)[0] for n in (30000, 1, 0, 2500)]
    streams[1] = b"@"
    eng = _engine(4)
    got = _encode(eng, streams, random.Random(3))
    again = _encode(eng, streams, random.Random(4))
    assert got == again
    for blob, want in zip(got, streams):
        check_file(blob, want)
    assert got[2] == EOF_MEMBER


# ---- the splitter

def _split(inp, barcodes, outs, bgzf, **kw):
    from tagdigger_b200 import splitter
    with contextlib.redirect_stdout(io.StringIO()) as so:
        splitter.barcodeSplitter(inp, barcodes, outs, bgzf=bgzf, **kw)
    return so.getvalue()


def _both(inp, barcodes, tag, **kw):
    """Plain and BGZF split of one input: the BGZF files inflate to the plain ones and have the
    member cuts of their streams; stdout is the same.  Returns the BGZF files' bytes."""
    plain = ["%s_p%d.fq" % (tag, i) for i in range(len(barcodes))]
    comp = ["%s_z%d.fq.gz" % (tag, i) for i in range(len(barcodes))]
    out_p = _split(inp, barcodes, plain, False, **kw)
    out_z = _split(inp, barcodes, comp, True, **kw)
    assert out_p == out_z
    blobs = []
    for p, z in zip(plain, comp):
        want = open(p, "rb").read()
        blob = open(z, "rb").read()
        check_file(blob, want)
        blobs.append(blob)
    return blobs


def test_splitter_golden_bgzf(in_tmp):
    for i, case in enumerate(load_golden("splitter.json")):
        materialize(case["files"], in_tmp)
        inp, barcodes, outs = case["args"]
        kw = dict(case["kwargs"])
        kw["adapter"] = [tuple(x) for x in kw["adapter"]]
        comp = ["g%d_%d.gz" % (i, k) for k in range(len(outs))]
        _split(inp, barcodes, comp, True, **kw)
        for name, z in zip(outs, comp):
            check_file(open(z, "rb").read(), base64.b64decode(case["outfiles"][name]))


@pytest.mark.parametrize("name", sorted(hostio.adapters))
def test_splitter_oracle_cases_bgzf(name, in_tmp, monkeypatch):
    from tagdigger_b200 import splitter
    monkeypatch.setattr(splitter, "BLOCK_READS", 700)
    rng = random.Random(len(name) * 7 + 1)
    adapter = hostio.adapters[name]
    cutsite = "TGCAG" if name.startswith("PstI") else "TGCAT"
    barcodes = []
    while len(barcodes) < 9:
        b = "".join(rng.choice("ACGT") for _ in range(rng.randint(4, 9)))
        pat = b + cutsite
        if not any(p.startswith(pat) or pat.startswith(p) for p in (x + cutsite for x in barcodes)):
            barcodes.append(b)
    for newline, gz, maxreads in (("\n", False, 500000000), ("\r\n", True, 1234), ("\n", False, 1)):
        text = _make_input(rng, barcodes, cutsite, adapter, 3000, newline)
        inp = "in.fq.gz" if gz else "in.fq"
        data = text.encode("utf-8")
        with open(inp, "wb") as fh:
            fh.write(gzip.compress(data) if gz else data)
        _both(inp, barcodes, "c", cutsite=cutsite, adapter=adapter, maxreads=maxreads)


def _shapes(rng):
    barcodes = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA"]
    base = _make_input(rng, barcodes, "TGCAG", ADAPTER, 1500) * 12               # 18,000 reads: several members per file
    recs = base.split("\n")
    recs = ["\n".join(recs[i:i + 4]) + "\n" for i in range(0, len(recs) - 1, 4)]
    for i in range(100, len(recs), 4011):                                      # non-ASCII: host blocks mid-stream
        c1, s, c2, q = recs[i].split("\n")[:4]
        recs[i] = "\n".join([c1, s[:12] + "é" + s[12:], c2, "ß" + q]) + "\n"
    mixed = "".join(recs)
    return barcodes, [("lf", base, {}), ("crlf", base.replace("\n", "\r\n"), {}), ("cr", base.replace("\n", "\r"), {}),
                      ("non-ascii", mixed, {}), ("maxreads", mixed, {"maxreads": 12345}), ("gz", base, {"gz": True})]


def test_splitter_bgzf_block_sizes(in_tmp, monkeypatch):
    """Block sizes of 1,500 B, 40 kB and 64 MiB give the same compressed files, byte for byte."""
    from tagdigger_b200 import splitter
    barcodes, cases = _shapes(random.Random(5))
    for label, text, kw in cases:
        inp = "in.fq.gz" if kw.pop("gz", False) else "in.fq"
        data = text.encode("utf-8")
        with open(inp, "wb") as fh:
            fh.write(gzip.compress(data, 1) if inp.endswith("gz") else data)
        seen = None
        for block_bytes in (1500, 40000, 64 << 20):
            monkeypatch.setattr(splitter, "BLOCK_BYTES", block_bytes)
            monkeypatch.setattr(splitter, "BLOCK_READS", 3000)
            blobs = _both(inp, barcodes, "s", adapter=ADAPTER, **kw)
            if seen is None:
                seen = blobs
                assert all(len(gzip.decompress(b)) > 2 * BLOCK for b in blobs), label
            assert blobs == seen, (label, block_bytes)


def test_splitter_bgzf_needs_gz_names(in_tmp):
    open("in.fq", "w").write(_make_input(random.Random(1), ["ACGTA"], "TGCAG", ADAPTER, 10))
    with pytest.raises(ValueError):
        _split("in.fq", ["ACGTA", "GGAT"], ["a.fq.gz", "b.fastq"], True, adapter=ADAPTER)
    assert not os.path.exists("a.fq.gz") and not os.path.exists("b.fastq")
    _split("in.fq", ["ACGTA", "GGAT"], ["a.fq.GZ", "b.gz"], True, adapter=ADAPTER)
    assert os.path.exists("b.gz")


def test_cli_bgzf_flag(in_tmp):
    p = barcode_splitter_script.build_parser()
    assert p.parse_args(["-b", "k.csv", "-a", "PstI-MspI-Hall"]).bgzf is False
    assert p.parse_args(["-b", "k.csv", "-a", "PstI-MspI-Hall", "--bgzf"]).bgzf is True
    barcodes = ["ACGTA", "TTGCAC", "GGAT"]
    open("in.fq", "w").write(_make_input(random.Random(2), barcodes, "TGCAG", ADAPTER, 2000))
    with open("key.csv", "w") as fh:
        fh.write("Input File,Barcode,Output File\n")
        for i, b in enumerate(barcodes):
            fh.write("in.fq,%s,z%d.fq.gz\n" % (b, i))
    with contextlib.redirect_stdout(io.StringIO()):
        assert barcode_splitter_script.main(["-b", "key.csv", "-a", "PstI-MspI-Hall", "--bgzf"]) == 0
    plain = ["p%d.fq" % i for i in range(3)]
    _split("in.fq", barcodes, plain, False, adapter=ADAPTER)
    for i in range(3):
        check_file(open("z%d.fq.gz" % i, "rb").read(), open(plain[i], "rb").read())


def test_count_split_bgzf_files(in_tmp, monkeypatch):
    """count_files over the BGZF split files equals count_files over the plain ones, cell by cell, with
    the device BGZF feed (files of >= 8 MiB) and with the host feed."""
    from tagdigger_b200 import counting, synth
    nrng = np.random.default_rng(4)
    bcs = synth.make_barcodes(2, nrng)
    _, _, seqs = synth.make_marker_pairs(300, nrng)
    tags = [s for p in seqs for s in p]
    fq, _ = synth.make_fastq(200000, bcs, tags, nrng)
    open("in.fq", "wb").write(fq)
    plain = ["p%d.fq" % i for i in range(2)]
    comp = ["z%d.fq.gz" % i for i in range(2)]
    _split("in.fq", bcs, plain, False)
    _split("in.fq", bcs, comp, True)
    assert all(os.path.getsize(z) >= 8 << 20 for z in comp), [os.path.getsize(z) for z in comp]

    def count(files):
        keys = {f: [[""], ["S%d" % i]] for i, f in enumerate(files)}
        with contextlib.redirect_stdout(io.StringIO()):
            return np.asarray(counting.count_files(keys, tags, "TGCAG", as_array=True)[1])

    want = count(plain)
    assert want.sum() > 0
    eng = counting.get_engine(0)
    for z in comp:
        got = count([z])
        assert eng.last_file_info()["mode"] == 0                    # the device feed inflated the file
        assert (got[0] == want[comp.index(z)]).all()
    assert (count(comp) == want).all()
    monkeypatch.setenv("TDG_GZDEV", "0")
    assert (count(comp) == want).all()
