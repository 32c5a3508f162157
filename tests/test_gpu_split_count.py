"""Counting adapter-trimmed reads in one GPU pass: count_files(..., adapter=...) and tagdigger_script
--adapter against the reference's recorded two-stage flow, against the oracle's two-stage composition
(tests/split_count_check.py), and against the GPU's own two-stage run (barcodeSplitter to files, then
count_files with blank barcodes)."""

import base64
import contextlib
import gzip
import io
import os
import random

import numpy as np
import pytest

from conftest import load_golden, materialize
from split_count_check import make_reads, make_tags, two_stage
from tagdigger_b200 import _native, counting, hostio, matchset, splitter, tagdigger_script

pytestmark = pytest.mark.gpu

FLOW = load_golden("flow.json")["cases"][0]
PSTI_BARCODES = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA", "AACCGT"]


@pytest.fixture
def small_blocks(monkeypatch):
    """Several device blocks and several host batches per file."""
    monkeypatch.setattr(splitter, "BLOCK_BYTES", 40000)
    monkeypatch.setattr(splitter, "BLOCK_READS", 300)


@pytest.fixture
def library():
    rng = random.Random(11)
    tags = make_tags(rng, "TGCAG", 60)
    return rng, tags, make_reads(rng, PSTI_BARCODES, "TGCAG", tags, hostio.adapters["PstI-MspI-Hall"], 2500)


def write_input(name, text):
    data = text.encode("utf-8")
    with open(name, "wb") as fh:
        fh.write(gzip.compress(data) if name.endswith("gz") else data)


def check(texts, key, tags, cutsite, adapter_name, split_cutsite=None, split_maxreads=500000000, label=""):
    """The one-pass count equals the oracle's two-stage composition (matrix and totals) and the GPU's
    two-stage run (matrix and tag hits).  Returns the one-pass matrix."""
    for f, text in texts.items():
        write_input(f, text)
    adapter = hostio.adapters[adapter_name]
    s1 = hostio.enzymes[adapter_name[:adapter_name.find("-")]] if split_cutsite is None else split_cutsite
    got_tot = {}
    with contextlib.redirect_stdout(io.StringIO()):
        samples, got = counting.count_files(key, tags, cutsite, adapter=adapter_name, split_cutsite=split_cutsite,
                                            split_maxreads=split_maxreads, totals=got_tot, as_array=True)
        want_samples, want, want_tot = two_stage(texts, key, tags, cutsite, adapter, s1, split_maxreads)
    assert samples == want_samples, label
    assert np.array_equal(got, np.asarray(want, dtype=np.int32).reshape(got.shape)), label
    assert got_tot == want_tot, label
    # the GPU two-stage run: split files named so that their sorted order is (input file, barcode)
    count_key = {}
    with contextlib.redirect_stdout(io.StringIO()):
        for f in sorted(key):
            outs = ["%s.split%03d.fq" % (f, i) for i in range(len(key[f][0]))]
            splitter.barcodeSplitter(f, key[f][0], outs, cutsite=s1, adapter=adapter, maxreads=split_maxreads)
            for o, sample in zip(outs, key[f][1]):
                count_key[o] = [[""], [sample]]
        stage2_tot = {}
        samples2, two = counting.count_files(count_key, tags, cutsite, totals=stage2_tot, as_array=True)
    assert samples2 == samples and np.array_equal(two, got), label
    for f in key:
        assert got_tot[f][3] == sum(t[2] for o, t in stage2_tot.items() if o.startswith(f + ".split")), label
    return got


def test_golden_flow_in_one_pass(in_tmp):
    """The recorded flow's library counted with --adapter gives the reference's two-stage CSVs."""
    materialize(FLOW["files"], in_tmp)
    split = hostio.readBarcodeKeyfile("split_key.csv", forSplitter=True)
    count = hostio.readBarcodeKeyfile("count_key.csv")
    (lib, (barcodes, outputs)), = split.items()
    with open("fused_key.csv", "w") as fh:
        fh.write("File,Barcode,Sample\n" + "".join("%s,%s,%s\n" % (lib, b, count[o][1][0]) for b, o in zip(barcodes, outputs)))
    argv = list(FLOW["count_argv"])
    argv[argv.index("count_key.csv")] = "fused_key.csv"
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        assert tagdigger_script.main(argv + ["--adapter", "PstI-MspI-Hall"]) == 0
    for name, b64 in FLOW["outfiles"].items():
        with open(name, "rb") as fh:
            assert fh.read() == base64.b64decode(b64), name
    assert not any(os.path.exists(o) for o in outputs)                # no split files
    line, = [ln for ln in out.getvalue().splitlines() if ln.startswith(lib + ": ")]
    assert line.startswith(lib + ": Reads: ") and " Clipped on 3' end: " in line and " With tag: " in line


@pytest.mark.parametrize("name", sorted(hostio.adapters))
def test_adapter_sets(name, in_tmp, small_blocks):
    """Every adapter set, Poland's overlap fallback included; the trim removes tag hits that the
    untrimmed reads have."""
    rng = random.Random(len(name) * 13)
    site = hostio.enzymes[name[:name.find("-")]]
    barcodes = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA"]
    tags = make_tags(rng, site, 50)
    text = make_reads(rng, barcodes, site, tags, hostio.adapters[name], 3000)
    key = {"lib.fq": [barcodes, ["S0", "S1", "S2", "S0"]]}
    got = check({"lib.fq": text}, key, tags, site, name, label=name)
    with contextlib.redirect_stdout(io.StringIO()):
        _, untrimmed = counting.count_files(key, tags, site, as_array=True)
    assert (got <= untrimmed).all() and (got < untrimmed).any() and got.sum() > 100


@pytest.mark.parametrize("block_bytes", [1500, 40000, 64 << 20])
def test_text_shapes_and_blocks(in_tmp, monkeypatch, library, block_bytes):
    """Block edges, newline conventions, gzip, text the host has to cut (non-ASCII), blank lines that
    shift the record phase, partial records, empty input and split_maxreads."""
    monkeypatch.setattr(splitter, "BLOCK_BYTES", block_bytes)
    monkeypatch.setattr(splitter, "BLOCK_READS", 300)
    rng, tags, text = library
    key = lambda f: {f: [PSTI_BARCODES, ["A", "B", "C", "A", "D"]]}      # noqa: E731
    recs = text.split("\n")
    recs = ["\n".join(recs[i:i + 4]) + "\n" for i in range(0, len(recs) - 1, 4)]
    mixed = list(recs)
    for i in range(100, len(mixed), 311):
        c1, s, c2, q = mixed[i].split("\n")[:4]
        mixed[i] = "\n".join([c1, s[:20] + "é" + s[20:], c2, "ß" + q if i % 2 else q]) + "\n"
    mixed = "".join(mixed)
    shapes = [("lf", "in.fq", text), ("crlf", "in.fq", text.replace("\n", "\r\n")), ("cr", "in.fq", text.replace("\n", "\r")),
              ("gzip", "in.fq.gz", text.replace("\n", "\r\n")), ("non-ascii", "in.fq", mixed),
              ("blank line shifts the phase", "in.fq", "".join(recs[:40]) + "\n" + "".join(recs[40:])),
              ("partial record", "in.fq", text + "@x\nACGTATGCAGTT\n"), ("no final newline", "in.fq", text[:-1]),
              ("empty", "in.fq", "")]
    for label, f, t in shapes:
        check({f: t}, key(f), tags, "TGCAG", "PstI-MspI-Hall", label=label)
    for m in (1, 1234):
        check({"in.fq": mixed}, key("in.fq"), tags, "TGCAG", "PstI-MspI-Hall", split_maxreads=m, label="maxreads %d" % m)


def test_stage_two_cut_sites(in_tmp, small_blocks, library):
    """Stage 2 with no cut site (-e None: any A/C/G/T starts the tag), and ApeKI's two sites after a
    split without cut site -- blanks behind the barcode surface at the start of the trimmed line."""
    rng, tags, text = library
    key = {"lib.fq": [PSTI_BARCODES, ["A", "B", "C", "D", "E"]]}
    got = check({"lib.fq": text}, key, tags, "", "PstI-MspI-Hall", label="-e None")
    assert got.sum() > 100
    ape = make_tags(rng, "CAGC", 20) + make_tags(rng, "CTGC", 20)           # ApeKI (CWGC): tags start at a site
    reads = make_reads(rng, PSTI_BARCODES, "", ape, hostio.adapters["PstI-MspI-Hall"], 2000)
    recs = reads.split("\n")
    for i in range(1, len(recs), 24):                                   # "barcode  CAGC..." on some sequence lines
        for bc in PSTI_BARCODES:
            if recs[i].startswith(bc):
                recs[i] = bc + "  " + recs[i][len(bc):]
                break
    got = check({"lib.fq": "\n".join(recs)}, key, ape, "CWGC", "PstI-MspI-Hall", split_cutsite="", label="ApeKI")
    assert got.sum() > 100


def test_blank_barcode_and_shared_samples(in_tmp, small_blocks, library):
    """A blank barcode trims pre-split files; two inputs whose barcodes share samples merge by sample."""
    rng, tags, text = library
    check({"one.fq": text}, {"one.fq": [[""], ["S"]]}, tags, "TGCAG", "PstI-MspI-Clark", label="blank barcode")
    other = make_reads(rng, ["CCATG", "ACGTA", "GTTAC"], "TGCAG", tags, hostio.adapters["PstI-MspI-Clark"], 1500)
    key = {"a.fq": [PSTI_BARCODES, ["S1", "S2", "S3", "S4", "S5"]], "b.fq.gz": [["CCATG", "ACGTA", "GTTAC"], ["S3", "S6", "S1"]]}
    got = check({"a.fq": text, "b.fq.gz": other}, key, tags, "TGCAG", "PstI-MspI-Clark", label="two files")
    assert got.shape[0] == 6


BOUND = 120


def _fused(eng, path, barcodes, tags):
    plan = matchset.plan([""], tags, "TGCAG")
    eng.set_tags(plan.tags.patterns, plan.tags.index, any_base=plan.tags.any_base)
    eng.set_matrix(3, plan.ntags)
    tot = splitter.count_trimmed_file(eng, path, barcodes, [0, 2, 1, 0, 2], plan, adapter=hostio.adapters["PstI-MspI-Hall"])
    return eng.read_matrix().tobytes(), tot


def test_allocation_failure_sweep(in_tmp, monkeypatch, library):
    """TDG_FAIL_ALLOC=k over one file counted in one pass, device blocks and host batches both: every
    failure is TDG_ERR_NOMEM, and the file counted again equals the run without a failure."""
    monkeypatch.setattr(splitter, "BLOCK_BYTES", 60000)
    monkeypatch.setattr(splitter, "BLOCK_READS", 200)
    rng, tags, text = library
    recs = text.split("\n")
    recs[4 * 700 + 1] = recs[4 * 700 + 1] + "é"                   # one block goes to the host
    write_input("in.fq", "\n".join(recs))
    monkeypatch.delenv("TDG_FAIL_ALLOC", raising=False)
    eng = _native.Engine(0)
    want = _fused(eng, "in.fq", PSTI_BARCODES, tags)
    eng.close()
    for k in range(1, BOUND + 1):
        monkeypatch.setenv("TDG_FAIL_ALLOC", str(k))
        eng = _native.Engine(0)
        failed = False
        try:
            got = _fused(eng, "in.fq", PSTI_BARCODES, tags)
        except _native.TdgError as e:
            assert e.code == _native.TDG_ERR_NOMEM and "simulated" in e.message, (k, e.code, e.message)
            failed = True
            got = _fused(eng, "in.fq", PSTI_BARCODES, tags)
        eng.close()
        assert got == want, k
        if not failed:
            break
    else:
        pytest.fail("every one of %d runs met a simulated failure" % BOUND)
    assert k > 10, k
