"""The oracle (oracle/tagdigger_oracle.py) against the golden vectors recorded
from the reference, and -- when it is staged in oracle/_ref -- against the live
reference on fresh random inputs.  CPU only."""

import base64
import contextlib
import io
import random

import numpy as np
import pytest

from conftest import NO_REFERENCE, file_bytes, have_reference, import_reference, load_golden, materialize
from oracle import tagdigger_oracle as orc

FIND = load_golden("find_tags.json") + load_golden("find_tags_text.json")     # + text-mode cases (UTF-8, maxreads stop)


def _call(fn, *a, **kw):
    try:
        return fn(*a, **kw), None
    except BaseException as e:  # noqa: BLE001
        return None, [type(e).__name__, str(e)]


@pytest.mark.parametrize("i", range(len(FIND)))
def test_find_tags_fastq_golden(i, in_tmp):
    case = FIND[i]
    materialize(case["files"], in_tmp)
    ret, exc = _call(orc.find_tags_fastq, *case["args"], **case["kwargs"])
    if case["exc"] is not None:
        assert exc is not None and exc[0] == case["exc"][0], (exc, case["exc"])
        if case["exc"][0] == "AssertionError":
            assert exc[1] == case["exc"][1]
    else:
        assert exc is None, exc
        assert ret == case["ret"]


def test_small_functions_golden():
    for case in load_golden("small_functions.json"):
        f, a = case["func"], case["args"]
        if f == "enumerate_cut_sites":
            assert orc.expand_cut_site(*a) == case["ret"]
        elif f == "combine_barcode_and_cutsite":
            ret, exc = _call(orc.barcode_patterns, *a)
            assert (exc[0] if exc else None) == (case["exc"][0] if case["exc"] else None)
            assert ret == case["ret"]
        elif f == "reverseComplement":
            assert orc.reverse_complement(*a) == case["ret"]
        elif f == "sanitizeTags":
            ret, exc = _call(orc.sanitize_tags, a[0][0], a[0][1])
            if case["exc"]:
                assert exc and exc[0] == case["exc"][0]
            else:
                assert [ret[0], ret[1]] == case["ret"]
        elif f == "extractMarkers":
            ret, exc = _call(orc.extract_markers, *a)
            assert (exc is None) == (case["exc"] is None)
            assert ret == case["ret"]
        elif f == "combineReadCounts":
            assert orc.combine_read_counts(*a) == case["ret"]
        elif f == "writeCounts" and case["exc"] is None:
            got = orc.counts_csv_bytes(a[1], a[2], a[3])
            assert got == base64.b64decode(case["outfiles"][a[0]])
        elif f == "writeDiploidGeno" and case["outfiles"].get(a[0]):
            got = orc.diploid_geno_csv_bytes(a[1], a[2], a[3])
            assert got == base64.b64decode(case["outfiles"][a[0]])


def test_trim_decision_golden():
    for case in load_golden("trim.json"):
        adapter = [tuple(x) for x in case["adapter"]]
        tables = orc.adapter_tables(adapter, case["barcodes"])
        assert [t[1] for t in tables] == case["indices"]
        full0 = adapter[0][0].replace("^", "")
        full1 = adapter[1][0].replace("^", "")
        for s, b, st, want in zip(case["seqs"], case["barindex"], case["searchstart"], case["slice2"]):
            assert orc.find_adapter_seq(s, tables[b], full0, full1, st) == want


def test_splitter_golden(in_tmp):
    for case in load_golden("splitter.json"):
        materialize(case["files"], in_tmp)
        inp, barcodes, outs = case["args"]
        kw = case["kwargs"]
        adapter = [tuple(x) for x in kw["adapter"]]
        bufs = [io.StringIO() for _ in barcodes]
        with orc.open_text(inp) as con:
            for b, lines, _ in orc.split_records(con, barcodes, kw["cutsite"], adapter, kw["maxreads"]):
                bufs[b].write("".join(l + "\n" for l in lines))
        for name, buf in zip(outs, bufs):
            assert buf.getvalue().encode() == base64.b64decode(case["outfiles"][name])


# ---- live differential tests (where the reference is staged in oracle/_ref) --

needs_ref = pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)


def _rand_seq(r, n):
    return "".join(r.choice("ACGT") for _ in range(n))


@needs_ref
@pytest.mark.parametrize("seed", range(60))
def test_trie_rules_live(seed):
    """Random pattern lists full of duplicates and prefix overlaps: same index,
    same AssertionError text, same lookups."""
    ref = import_reference()
    r = random.Random(seed)
    pool = [_rand_seq(r, r.randint(1, 5)) for _ in range(6)]
    pats = []
    for _ in range(r.randint(1, 10)):
        p = r.choice(pool)
        if r.random() < 0.4:
            p += _rand_seq(r, r.randint(1, 3))
        pats.append(p)
    numseq = r.choice([len(pats), max(1, len(pats) // 2)])
    want, wexc = _call(ref.build_sequence_tree, [p for p in pats], numseq)
    got, gexc = _call(orc.build_trie, pats, numseq)
    assert (wexc is None) == (gexc is None)
    if wexc is not None:
        assert wexc == gexc
        return
    for _ in range(200):
        q = r.choice(pats)[:r.randint(0, 8)] + _rand_seq(r, r.randint(0, 4))
        if r.random() < 0.1:
            q = q[:1] + "N" + q[1:]
        assert orc.lookup(q, got) == ref.sequence_index_lookup(q, want), (pats, q)


@needs_ref
def test_synthetic_config1_shape_live(tmp_path):
    """20k reads of the config-1 shape through reference and oracle."""
    from tagdigger_b200 import synth
    ref = import_reference()
    rng = np.random.default_rng(5)
    bcs = synth.make_barcodes(24, rng)
    _, _, seqs = synth.make_marker_pairs(150, rng)
    tags = [s for p in seqs for s in p]
    fq, _ = synth.make_fastq(20000, bcs, tags, rng)
    path = str(tmp_path / "x.fq")
    with open(path, "wb") as fh:
        fh.write(fq)
    with contextlib.redirect_stdout(io.StringIO()):
        want = ref.find_tags_fastq(path, bcs, tags)
    assert orc.find_tags_fastq(path, bcs, tags) == want
    assert orc.find_tags_text(fq, bcs, tags) == want
