"""Trim decision (SURVEY.md 8(a) row A8): the host tables of tagdigger_b200/trimming.py
against the oracle's trie (CPU), and the CUDA decision (csrc/tdg_trim.cuh, through
tdg_set_trim / tdg_trim_batch) against the slice indices recorded from the reference's
findAdapterSeq (tests/golden/trim.json) and against the oracle on fresh reads (GPU)."""

import contextlib
import io
import random

import pytest

from conftest import NO_REFERENCE, have_reference, import_reference, load_golden
from helpers import rand_seq
from oracle import tagdigger_oracle as orc
from tagdigger_b200 import hostio, trimming

GOLD = load_golden("trim.json")


def tables_decide(seq, tables, b, start):
    """Evaluate the host tables the way the kernel does (test-side model, plain Python)."""
    site0, site1, a0, a1_all, cands = tables
    s = seq.upper()
    p0, p1 = s.find(site0, start), s.find(site1, start)
    if p0 != -1 or p1 != -1:
        if p1 == -1 or (p0 != -1 and p0 < p1):
            return p0 + len(site0)
        return p1 + len(site1)
    for which, length, idx in cands[b]:
        full = a1_all[b] if which else a0
        if length <= len(s) and s.endswith(full[:length]):
            return idx
    return 999


def make_reads(rng, adapter, barcodes, cutsite, n):
    full0 = adapter[0][0].replace("^", "")
    full1 = adapter[1][0].replace("^", "")
    a0 = adapter[0][0][:adapter[0][0].find("^")] + adapter[0][1]
    seqs, bars, starts = [], [], []
    for _ in range(n):
        b = rng.randrange(len(barcodes))
        bc = barcodes[b]
        a1 = adapter[1][0][:adapter[1][0].find("^")] + adapter[1][1].replace("[barcode]", hostio.reverseComplement(bc))
        insert = rand_seq(rng, rng.randint(0, 120))
        k = rng.random()
        if k < 0.35:
            tail = rng.choice([a0, a1])[:rng.randint(1, 75)]
        elif k < 0.45:
            tail = rng.choice([a0, a1]) + rand_seq(rng, rng.randint(1, 6))
        elif k < 0.6:
            tail = rng.choice([full0, full1]) + rand_seq(rng, rng.randint(0, 40))
        elif k < 0.7:
            tail = full0 + rand_seq(rng, rng.randint(0, 6)) + full1 + rand_seq(rng, 4)
        elif k < 0.8:
            tail = full1 + rand_seq(rng, rng.randint(0, 6)) + full0
        else:
            tail = rand_seq(rng, rng.randint(0, 40))
        s = (bc + cutsite + insert + tail)[:rng.choice([0, 3, 31, 32, 33, 60, 64, 100, 100, 150, 300])]
        w = rng.random()
        if s and w < 0.08:
            j = rng.randrange(len(s))
            s = s[:j] + rng.choice("Nn.") + s[j + 1:]
        elif w < 0.16:
            s = s.lower()
        seqs.append(s)
        bars.append(b)
        starts.append(rng.choice([len(bc) + len(cutsite), 0, 1, len(s), len(s) + 3]))
    return seqs, bars, starts


def random_barcodes(rng, n):
    out = set()
    while len(out) < n:
        out.add(rand_seq(rng, rng.randint(4, 9)))
    return sorted(out)


@pytest.mark.parametrize("name", sorted(hostio.adapters))
def test_tables_equal_oracle_trie(name):
    rng = random.Random(hash(name) & 0xFFFF)
    adapter = hostio.adapters[name]
    cutsite = "TGCAG" if name.startswith("PstI") else "TGCAT"
    barcodes = random_barcodes(rng, 12) + ["CTGCA", "TGCAG", "AGATC", "CCG", "GGCC"]      # collide with adapter starts
    with contextlib.redirect_stdout(io.StringIO()):
        tables = trimming.trim_tables(adapter, barcodes)
        want_tables = orc.adapter_tables(adapter, barcodes)
    full0, full1 = tables[0], tables[1]
    seqs, bars, starts = make_reads(rng, adapter, barcodes, cutsite, 1500)
    for s, b, st in zip(seqs, bars, starts):
        want = orc.find_adapter_seq(s.upper(), want_tables[b], full0, full1, st)
        assert tables_decide(s, tables, b, st) == want, (s, barcodes[b], st)


def test_tables_golden_model():
    for case in GOLD:
        adapter = [tuple(x) for x in case["adapter"]]
        assert hostio.adapters[case["adapter_name"]] == adapter      # recorded from the reference's adapters
        with contextlib.redirect_stdout(io.StringIO()):
            tables = trimming.trim_tables(adapter, case["barcodes"])
        for s, b, st, want in zip(case["seqs"], case["barindex"], case["searchstart"], case["slice2"]):
            assert tables_decide(s, tables, b, st) == want


@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
def test_fallback_messages_match_reference():
    ref = import_reference()
    rng = random.Random(5)
    for name in sorted(hostio.adapters):
        barcodes = random_barcodes(rng, 6) + ["CTGCA", "AGATC"]
        got, want = io.StringIO(), io.StringIO()
        with contextlib.redirect_stdout(got):
            trimming.trim_tables(hostio.adapters[name], barcodes)
        with contextlib.redirect_stdout(want):
            ref.build_adapter_tree(ref.adapters[name], barcodes)
        assert got.getvalue() == want.getvalue()
        assert hostio.adapters[name] == ref.adapters[name]


@pytest.mark.gpu
def test_trim_kernel_golden():
    from tagdigger_b200 import _native
    eng = _native.Engine(0)
    for case in GOLD:
        adapter = [tuple(x) for x in case["adapter"]]
        with contextlib.redirect_stdout(io.StringIO()):
            trimming.load_trim(eng, adapter, case["barcodes"])
        got = trimming.find_adapter_seqs(eng, case["seqs"], case["barindex"], case["searchstart"])
        assert got == case["slice2"], case["adapter_name"]
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(hostio.adapters))
def test_trim_kernel_against_oracle(name):
    from tagdigger_b200 import _native
    eng = _native.Engine(0)
    rng = random.Random(1000 + len(name))
    adapter = hostio.adapters[name]
    cutsite = "TGCAG" if name.startswith("PstI") else "TGCAT"
    barcodes = random_barcodes(rng, 40) + ["CTGCA", "TGCAG", "AGATC", "CCG"]
    with contextlib.redirect_stdout(io.StringIO()):
        full0, full1 = trimming.load_trim(eng, adapter, barcodes)
        want_tables = orc.adapter_tables(adapter, barcodes)
    seqs, bars, starts = make_reads(rng, adapter, barcodes, cutsite, 20000)
    want = [orc.find_adapter_seq(s.upper(), want_tables[b], full0, full1, st) for s, b, st in zip(seqs, bars, starts)]
    got = trimming.find_adapter_seqs(eng, seqs, bars, starts)
    bad = [i for i in range(len(want)) if got[i] != want[i]]
    assert not bad, (bad[:5], [(seqs[i], got[i], want[i]) for i in bad[:3]])
    assert trimming.find_adapter_seqs(eng, [], [], []) == []
    with pytest.raises(_native.TdgError):
        trimming.find_adapter_seqs(eng, ["ACGT"], [len(barcodes)], [0])
    eng.close()
