#!/usr/bin/env python3
"""Generate the golden vectors under tests/golden/ by RUNNING THE REFERENCE.

Run where a checkout of the reference exists (it imports its tagdigger_fun.py):

    TAGDIGGER_REFERENCE=<checkout> python tests/golden/make_golden.py

Every case is recorded as: the function called, the input files (text, or
base64 for gzip), the arguments, and what the reference did -- return value,
stdout, exception type/message and any files it wrote.  The tests replay the
cases against the oracle (oracle/), the host-side API mirror
(tagdigger_b200/tagdigger_fun.py) and, on a GPU, the CUDA path.

Nothing from the reference is copied: only its observable behaviour on these
inputs is stored.
"""

import base64
import contextlib
import gzip
import io
import json
import os
import random
import subprocess
import sys
import tempfile
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("TAGDIGGER_REFERENCE")
if not REF or not os.path.isfile(os.path.join(REF, "tagdigger_fun.py")):
    sys.exit("usage: TAGDIGGER_REFERENCE=<checkout of the original TagDigger> python tests/golden/make_golden.py")
sys.path.insert(0, REF)
sys.path.insert(0, REPO)
warnings.simplefilter("ignore")

import tagdigger_fun as ref  # noqa: E402  (the reference itself)


def jsonable(x):
    if isinstance(x, (list, tuple)):
        return [jsonable(v) for v in x]
    if isinstance(x, dict):
        return {str(k): jsonable(v) for k, v in x.items()}
    if isinstance(x, (set, frozenset)):
        return sorted(jsonable(v) for v in x)
    return x


def run_case(func, files=None, args=(), kwargs=None, outfiles=()):
    """Call ref.<func>(*args, **kwargs) in a scratch directory holding
    ``files``; record everything observable."""
    kwargs = kwargs or {}
    files = files or {}
    rec = {"func": func, "files": {}, "args": jsonable(list(args)), "kwargs": jsonable(kwargs)}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for name, content in files.items():
                if isinstance(content, bytes):
                    with open(name, "wb") as fh:
                        fh.write(content)
                    rec["files"][name] = {"b64": base64.b64encode(content).decode()}
                else:
                    with open(name, "w", newline="") as fh:
                        fh.write(content)
                    rec["files"][name] = {"text": content}
            out = io.StringIO()
            exc = None
            ret = None
            with contextlib.redirect_stdout(out):
                try:
                    ret = getattr(ref, func)(*args, **kwargs)
                except BaseException as e:  # noqa: BLE001 - we record whatever happens
                    exc = [type(e).__name__, str(e)]
            rec["ret"] = jsonable(ret)
            rec["stdout"] = out.getvalue()
            rec["exc"] = exc
            rec["outfiles"] = {}
            for name in outfiles:
                if os.path.exists(name):
                    with open(name, "rb") as fh:
                        rec["outfiles"][name] = base64.b64encode(fh.read()).decode()
                else:
                    rec["outfiles"][name] = None
        finally:
            os.chdir(cwd)
    return rec


def dump(name, cases):
    path = os.path.join(HERE, name)
    with open(path, "w") as fh:
        json.dump(cases, fh, indent=0, sort_keys=True)
        fh.write("\n")
    n = len(cases["cases"]) if isinstance(cases, dict) else len(cases)
    print("%-28s %4d cases %8d bytes" % (name, n, os.path.getsize(path)))


# ---------------------------------------------------------------------------
# helpers to build small, nasty FASTQ images
# ---------------------------------------------------------------------------

def rand_seq(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def prefix_free_barcodes(rng, n, cutsite, lo=3, hi=8):
    out, pats = [], []
    while len(out) < n:
        b = rand_seq(rng, rng.randint(lo, hi))
        p = b + cutsite
        if any(q.startswith(p) or p.startswith(q) for q in pats):
            continue
        out.append(b)
        pats.append(p)
    return out


def fastq_text(rng, reads, newline="\n", messy=True, final_newline=True):
    """``reads`` is a list of sequence strings.  Returns text."""
    rows = []
    for i, s in enumerate(reads):
        hdr = "@r%d:%s" % (i, rand_seq(rng, rng.randint(0, 12)))
        q = "".join(chr(rng.randint(35, 74)) for _ in range(len(s)))
        if messy and rng.random() < 0.2:
            q = rng.choice("@+") + q[1:]
        if messy and rng.random() < 0.1:
            s = s.lower()
        if messy and rng.random() < 0.1:
            s = rng.choice([" ", "\t", "  ", "\x0b", "\x0c", "\x1c", "\x1f "]) + s
        if messy and rng.random() < 0.1:
            s = s + rng.choice([" ", "\t", " \t "])
        plus = "+" if rng.random() < 0.8 else "+" + hdr[1:]
        rows.extend([hdr, s, plus, q])
    if isinstance(newline, list):
        txt = "".join(r + rng.choice(newline) for r in rows)
    else:
        txt = "".join(r + newline for r in rows)
    if not final_newline:
        txt = txt.rstrip("\r\n")
    return txt


def reads_for(rng, barcodes, cutsites, tags, offsets_in_tag, n, readlen=60):
    """Reads built from barcode+cutsite+tag with assorted damage."""
    out = []
    for _ in range(n):
        r = rng.random()
        b = rng.choice(barcodes)
        cs = rng.choice(cutsites)
        t = rng.choice(tags)
        body = t[offsets_in_tag:] if offsets_in_tag else t
        if r < 0.55:
            s = b + cs + body + rand_seq(rng, rng.randint(0, 20))
        elif r < 0.65:
            s = b + cs + rand_seq(rng, readlen)
        elif r < 0.75:
            s = rand_seq(rng, readlen)
        elif r < 0.85:
            s = b + cs + body
            k = rng.randrange(len(s))
            s = s[:k] + rng.choice("ACGTN.") + s[k + 1:]
        elif r < 0.92:
            s = (b + cs + body)[:rng.randint(0, len(b + cs + body))]
        else:
            s = b + cs + body[:-1]
        out.append(s)
    return out


# ---------------------------------------------------------------------------
# 1. find_tags_fastq
# ---------------------------------------------------------------------------

def cases_find_tags():
    cases = []
    rng = random.Random(20160)

    def add(fq, barcodes, tags, name="a.fq", **kw):
        files = {name: fq}
        c = run_case("find_tags_fastq", files, (name, barcodes, tags), kw)
        c["stdout"] = ""          # progress prints are not part of parity
        cases.append(c)

    # --- SURVEY Appendix A.4 known answers -------------------------------
    one = lambda s: "@h\n%s\n+\n%s\n" % (s, "I" * len(s))
    add(one("AACGTGCAGTGCAGAAAT"), ["AACG"], ["TGCAGAAA", "CCCC"])
    add(one("AACGTGCAGTGCAGAAAT"), ["AACG"], ["TGCAGAAA", "TGCAGCCCC"])
    add(one("aacgtgcagcccc") + one("  AACGTGCAGCCCC "), ["AACG"], ["TGCAGAAA", "CCCC"])
    add(one("AACGTGCAGCCNC") + one("AACGTGCAGCC"), ["AACG"], ["TGCAGAAA", "CCCC"])
    add(one("AACGTGCAGCCCC").replace("\n", "\r\n") * 2, ["AACG"], ["CCCC"])
    add(one("AACGTGCAGCCCC").replace("\n", "\r") * 2, ["AACG"], ["CCCC"])
    ape = one("AACGCAGCTTTT") + one("AACGCTGCTTTT")
    add(ape, ["AACG"], ["CAGCTTTT", "CTGCTTTT"], cutsite="CWGC")
    add(ape, ["AACG"], ["TTTT"], cutsite="CWGC")
    add(ape, [""], ["AACGC"], cutsite="")
    add("@x count=7\nAACGTGCAGCCCC\n+\nIIIIIIIIIIIII\n@y count=12\nAACGTGCAGCCCC\n+\nIIIIIIIIIIIII\n",
        ["AACG"], ["CCCC"], tassel_tagcount=True)
    add("@x nocount\nAACGTGCAGCCCC\n+\nIIIIIIIIIIIII\n", ["AACG"], ["CCCC"], tassel_tagcount=True)
    # --- degenerate files -------------------------------------------------
    add("", ["AACG"], ["CCCC"])
    add("@only header", ["AACG"], ["CCCC"])
    add("@h\nAACGTGCAGCCCC", ["AACG"], ["CCCC"])                 # no final newline
    add("@h\n\n+\n\n@h\n \t \n+\n\n", ["AACG"], ["CCCC"])         # empty / blank sequence lines
    add("\n\n\n\n" + one("AACGTGCAGCCCC"), ["AACG"], ["CCCC"])    # leading blank record
    add("\n" + one("AACGTGCAGCCCC") * 3, ["AACG"], ["CCCC"])      # phase shifted by one line
    add(one("AACGTGCAGCCCC") + "\r\n\r\r\n" + one("AACGTGCAGCCCC"), ["AACG"], ["CCCC"])
    add("@h\r" + "AACGTGCAGCCCC\r\n+\n" + "IIII\r" + one("AACGTGCAGCCCC"), ["AACG"], ["CCCC"])
    # sequence-like text on non-sequence lines must be ignored
    add("AACGTGCAGCCCC\nGGGG\nAACGTGCAGCCCC\nAACGTGCAGCCCC\n", ["AACG"], ["CCCC"])
    # control characters: stripped at the ends, fatal inside
    add(one("\x0b\x0cAACGTGCAGCCCC\x1c\x1d\x1e\x1f") + one("AACGTGC\x0bAGCCCC") + one("AACGTGCAGCC CC"),
        ["AACG"], ["CCCC"])
    # maxreads
    many = one("AACGTGCAGCCCC") * 7
    for mr in (1, 3, 2.5, 7, 100, 0):
        add(many, ["AACG"], ["CCCC"], maxreads=mr)
    # --- pattern-set rules (SURVEY A.2) -------------------------------------
    fq = one("AACGTGCAGCCCCAAAA") + one("AACGTGCAGCCCCTTTT") + one("AACGTGCAGGGGG")
    add(fq, ["AACG"], ["CCCC", "CCCC", "GGGG"])                  # duplicate tag: first wins
    add(fq, ["AACG"], ["CCCC", "CCCCAAAA", "GGGG"])              # shorter listed first: longer dropped
    add(fq, ["AACG"], ["CCCCAAAA", "CCCC", "GGGG"])              # longer listed first: AssertionError
    add(fq, ["AACG"], ["GGGG", "CCCCAAAA", "CCCCTTTT", "CCCC"])  # error deeper in the tree
    add(fq, ["AACG"], ["CCCCAAAA", "GGGG", "GGGGA", "CCCC"])     # silent drop + later error
    add(fq, ["AACG", "AACGT"], ["CCCC"])                         # barcode patterns overlap
    add(fq, ["AACGT", "AACG"], ["CCCC"])
    add(fq, ["AACG", "AACG"], ["CCCC"])                          # duplicate barcode (API level)
    add(fq, ["AACG"], [])                                        # no tags
    add(fq, ["AACG"], [""])                                      # the single empty tag
    add(fq, ["AACG"], ["", "CCCC"])
    add(fq, ["AACG"], ["CCCC", ""])
    add(fq, [], ["CCCC"])                                        # no barcodes
    add(fq, ["", "AACG"], ["CCCC"], cutsite="")
    add(fq, ["AACG", ""], ["TGCAGCCCC"], cutsite="")
    add(fq, ["AANG"], ["CCCC"])                                  # asserts
    add(fq, ["AACG"], ["CCNC"])
    add(fq, ["AACG"], ["CCCC"], cutsite="TGXAG")
    add(fq, ["aacg"], ["cccc", "gGgG"], cutsite="tgcag")         # case folding of inputs
    add(fq, ["AACG"], ["TGCAGCCCC", "TGCAGGGGG"])                # cut site stripped from tags
    add(fq, ["AACG"], ["TGCAGCCCC", "GGGG"])                     # mixed: nothing stripped
    add(fq, ["AACG"], ["TGCAG"])                                 # tag == cut site -> empty after strip
    add(fq, ["AACG"], ["TGCAG", "TGCAGCCCC"])
    # ambiguous cut sites with several letters
    rr = one("ACAGTCCCC") + one("ACGGTCCCC") + one("ACAATCCCC") + one("ACGACCCCC")
    add(rr, ["AC"], ["CCCC"], cutsite="RRT")
    add(rr, ["AC"], ["AGTCCCC", "GGTCCCC", "AATCCCC"], cutsite="RRT")
    add(rr, ["AC"], ["AGTCCCC", "CCCC"], cutsite="RRT")
    add(rr, ["AC", "GT"], ["CCCC"], cutsite="NNY")
    # gzip handling
    gzb = gzip.compress(many.encode())
    add(gzb, ["AACG"], ["CCCC"], name="a.fq.gz")
    add(gzb + gzip.compress((one("AACGTGCAGCCCC") * 2).encode()), ["AACG"], ["CCCC"], name="a.fastq.GZ")
    add(gzb, ["AACG"], ["CCCC"], name="notgz")                   # gz bytes, plain name
    add(many, ["AACG"], ["CCCC"], name="b.gz")                   # plain bytes, gz name
    cases.append(run_case("find_tags_fastq", {}, ("missing.fq", ["AACG"], ["CCCC"]), {}))

    # --- randomised small cases -----------------------------------------
    for seed in range(40):
        r = random.Random(1000 + seed)
        cutsite = r.choice(["TGCAG", "TGCAG", "CWGC", "", "CATGG", "TGCAGG", "GR"])
        sites = ref.enumerate_cut_sites(cutsite)
        nb = r.randint(1, 6)
        if r.random() < 0.15:
            barcodes = [""]
        else:
            barcodes = prefix_free_barcodes(r, nb, cutsite)
        ntag = r.randint(1, 24)
        with_cut = r.random() < 0.5
        tags = []
        while len(tags) < ntag:
            L = r.choice([4, 8, 17, 31, 32, 33, 59, 64, 65, 70, 129, 140])
            t = rand_seq(r, L)
            if with_cut:
                t = r.choice(sites) + t
            if any(u.startswith(t) or t.startswith(u) for u in tags):
                continue
            tags.append(t)
            if r.random() < 0.5 and len(tags) < ntag:     # an allelic partner
                k = r.randrange(len(t) - L, len(t))
                u = t[:k] + r.choice([c for c in "ACGT" if c != t[k]]) + t[k + 1:]
                if not any(v.startswith(u) or u.startswith(v) for v in tags):
                    tags.append(u)
        strip = with_cut and len(sites) == 1
        reads = reads_for(r, barcodes, sites, tags, len(cutsite) if with_cut else 0,
                          r.randint(20, 120))
        nlstyle = r.choice(["\n", "\n", "\r\n", "\r", ["\n", "\r\n", "\r"]])
        fq = fastq_text(r, reads, newline=nlstyle, final_newline=r.random() < 0.7)
        kw = {"cutsite": cutsite}
        if r.random() < 0.2:
            kw["maxreads"] = r.randint(1, len(reads))
        if r.random() < 0.3:
            add(gzip.compress(fq.encode()), barcodes, tags, name="r%d.fastq.gz" % seed, **kw)
        else:
            add(fq, barcodes, tags, name="r%d.fq" % seed, **kw)
    return cases


# ---------------------------------------------------------------------------
# 2. small pure functions
# ---------------------------------------------------------------------------

def cases_small():
    cases = []
    for cs in ["TGCAG", "CWGC", "RY", "NN", "", "BDHV", "ARYKMSWA", "GCNGC", "YR"]:
        cases.append(run_case("enumerate_cut_sites", {}, (cs,)))
    cases.append(run_case("combine_barcode_and_cutsite", {}, (["AACG", "ttg", ""], "tgcag")))
    cases.append(run_case("combine_barcode_and_cutsite", {}, (["AANG"], "TGCAG")))
    cases.append(run_case("combine_barcode_and_cutsite", {}, (["AACG"], "CWGC")))
    for s in ["ACGTTGCA", "", "ACGTN", "acgt", "AAAC"]:
        cases.append(run_case("reverseComplement", {}, (s,)))
    # sanitizeTags (mutates and returns its argument)
    san = [
        [["M1_0", "M1_1", "M2_0", "M2_1"], ["ACGT", "ACGA", "TTTT", "TTTA"]],
        [["M1_0", "M1_1", "M2_0", "M2_1"], ["ACGT", "ACGA", "ACGTT", "TTTA"]],
        [["TP1_0", "TP1_1", "TP10_0", "TP10_1", "TP2_0"], ["ACG", "TTT", "GGGG", "CCCC", "ACGT"]],
        [["A_0", "B_0", "C_0"], ["ACGT", "ACGT", "GG"]],
        [["A_0", "B_0", "C_0", "D_0"], ["AC", "ACG", "ACGT", "T"]],
        [["noUnderscore", "X_1"], ["AC", "ACG"]],
        [["A_0"], ["ACGT"]],
        [[], []],
        [["A_0", "B_0"], ["", "ACGT"]],
    ]
    for s in san:
        cases.append(run_case("sanitizeTags", {}, (s,)))
    # extractMarkers
    for names in [["M1_A_0", "M1_C_1", "M2_0", "M3_x_y_2", "M2_1"], ["a_0", "a_0"], ["plain", "plain2_1"], []]:
        cases.append(run_case("extractMarkers", {}, (names,)))
    # combineReadCounts
    bck = {"b.fq": [["AA", "CC"], ["s1", "s2"]], "a.fq": [["GG", "TT", "AC"], ["s2", "s3", "s3"]]}
    cd = {"b.fq": [[1, 2, 3], [4, 5, 6]], "a.fq": [[10, 20, 30], [40, 50, 60], [7, 8, 9]]}
    cases.append(run_case("combineReadCounts", {}, (cd, bck)))
    bck2 = {"x.fq": [[""], ["only"]]}
    cases.append(run_case("combineReadCounts", {}, ({"x.fq": [[5, 0]]}, bck2)))
    # writeCounts / writeDiploidGeno
    counts = [[0, 3, 1, 0], [2, 2, 0, 0], [0, 0, 0, 9]]
    sams = ["s,1", 'he said "hi"', "plain"]
    tn = ["M1_A_0", "M1_C_1", "M2_G_0", "M2_T_1"]
    cases.append(run_case("writeCounts", {}, ("out.csv", counts, sams, tn), outfiles=["out.csv"]))
    cases.append(run_case("writeDiploidGeno", {}, ("gen.csv", counts, sams, tn), outfiles=["gen.csv"]))
    cases.append(run_case("writeDiploidGeno", {}, ("gen.csv", counts, sams, ["M1_0", "M1_1", "M2_0", "M2_2"]),
                          outfiles=["gen.csv"]))
    cases.append(run_case("writeCounts", {}, ("out.csv", counts, sams[:2], tn), outfiles=["out.csv"]))
    # readMarkerNames
    cases.append(run_case("readMarkerNames", {"k.txt": "TP276\n TP1003 ,\n\n,,\nTP1206"}, ("k.txt",)))
    cases.append(run_case("readMarkerNames", {}, ("missing.txt",)))
    # isFastq
    fq = "@h\nACGTN\n+\nIIIII\n"
    cases.append(run_case("isFastq", {"a.fq": fq}, ("a.fq",)))
    cases.append(run_case("isFastq", {"a.fq.gz": gzip.compress(fq.encode())}, ("a.fq.gz",)))
    cases.append(run_case("isFastq", {"a.fq": ">h\nACGT\n+\nIIII\n"}, ("a.fq",)))
    cases.append(run_case("isFastq", {"a.fq": "@h\nACGU\n+\nIIII\n"}, ("a.fq",)))
    cases.append(run_case("isFastq", {"a.fq": "@h\nACGT\n-\nIIII\n"}, ("a.fq",)))
    cases.append(run_case("isFastq", {"a.fq": "@h\nacgtn\n+\n"}, ("a.fq",)))
    cases.append(run_case("isFastq", {}, ("missing.fq",)))
    cases.append(run_case("isFastq", {"a.fq": ""}, ("a.fq",)))
    cases.append(run_case("isFastq", {"a.fq": "@h\nACGT\n"}, ("a.fq",)))
    return cases


# ---------------------------------------------------------------------------
# 3. key file + tag readers
# ---------------------------------------------------------------------------

UNEAK = """>TP276_query_64
TGCAGAAAAAAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT
>TP276_hit_64
TGCAGAAACAAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT
>TP539_query_64
TGCAGAAAAAAACTTGAGAAAGGCCGTACTTTTAAAGTGTATTATAGAAAAATCTTAGGTGCAT
>TP539_hit_64
TGCAGAAATAAACTTGAGAAAGGCCGTACTTTTAAAGTGTATTATAGAAAAATCTTAGGTGCAT
"""

MERGED = """Marker name,Tag sequence,
TP276,TGCAGAAA[A/C]AAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT,
TP539,TGCAGAAA[A/T]AAACTTGAGAAAGGCCGTACTTTTAAAGTGTATTATAGAAAAATCTTAGGTGCAT,
Mrkr2010,ACGTAAACGATA[AAG/GAC]TACGATAAATTT,
Mrkr2011,GGATAAC[CAC/TAC/TAT]GGATTA,
Mrkr2012,CTCCAAGACCT[AG/C-]TTTTACGGG,
"""

COLUMNS = """Marker name,Tag sequence 0,Tag sequence 1,
TP276,TGCAGAAAAAAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT,TGCAGAAACAAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT,
TP539,TGCAGAAAAAAACTTGAGAAAGGCCGTACTTTTAAAGTGTATTATAGAAAAATCTTAGGTGCAT,TGCAGAAATAAACTTGAGAAAGGCCGTACTTTTAAAGTGTATTATAGAAAAATCTTAGGTGCAT,
"""

ROWS = """Marker name,Allele name,Tag sequence,
TP276,0,TGCAGAAAAAAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT,
TP276,1,TGCAGAAACAAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT,
Mrker2035,dom,AGCTAGACTAGGGTTACCAGTACTTACCGATACATTAAAGCATCAT,
Mrker4050,0,AGTAGGGAAAGGCCGGTAAGGCAACTAAA,
Mrker4050,1,AGTAGGGAGAGGCCGGTAAGGCAACTAAA,
Mrker4050,2,AGTAGGGAAAGGCCGGCAAGGCAACTAAA,
"""


def stacks_files(version=1):
    """A tiny Stacks catalog (tags/snps/alleles) in the v1 or v2 column layout."""
    loci = {
        "1": ("TGCAGAACCGTTAGGCATTACGGATCAGGT", [8, 20], ["AC", "GT"]),
        "2": ("TGCAGTTTTGGGCCCAAATTTGGGCCCAAA", [], [""]),
        "3": ("TGCAGCATCATCATCATCATCATCATCATC", [10], ["A", "G", "T"]),
        "4": ("TGCAGNNACGTACGTACGTACGTACGTACG", [12], ["A", "C"]),
        "7": ("TGCAGGGACGTACGTACGAACGTACGTACG", [29], ["G", "A"]),
    }
    tags, snps, alle = ["# comment line\tx"], ["# c"], ["# c"]
    for lid, (seq, pos, haps) in loci.items():
        if version == 1:
            tags.append("\t".join(["0", "1", lid, "", "0", "+", "consensus", "0", "", seq, "0", "0", "0"]))
            for p in pos:
                snps.append("\t".join(["0", "1", lid, str(p), "E", "0", "A", "C", "-", "-"]))
            for h in haps:
                alle.append("\t".join(["0", "1", lid, h, "50.0", "10"]))
        else:
            tags.append("\t".join(["0", lid, "", "0", "+", seq, "0", "0"]))
            for p in pos:
                snps.append("\t".join(["0", lid, str(p), "E", "0", "A", "C"]))
            for h in haps:
                alle.append("\t".join(["0", lid, h, "50.0", "10"]))
    j = lambda rows: "\n".join(rows) + "\n"
    return j(tags), j(snps), j(alle)


SAM = "\n".join([
    "@HD\tVN:1.0\tSO:unsorted",
    "@SQ\tSN:chr01\tLN:43270923",
    "@SQ\tSN:Chromosome_2\tLN:35937250",
    "@SQ\tSN:3\tLN:999",
    "@PG\tID:bowtie2",
    "tagSeq=A\t0\tchr01\t1000\t42\t20M\t*\t0\t0\tTGCAGAAAACCCCGGGGTTT\t*",
    "tagSeq=B\t0\tchr01\t1000\t42\t20M\t*\t0\t0\tTGCAGAAAACCCTGGGGTTT\t*",
    "tagSeq=C\t16\tchr01\t2000\t42\t20M\t*\t0\t0\tAAACCCCGGGGTTTTCTGCA\t*",
    "tagSeq=D\t16\tchr01\t2000\t42\t20M\t*\t0\t0\tAAACCCCGGTGTTTTCTGCA\t*",
    "tagSeq=E\t4\t*\t0\t0\t*\t*\t0\t0\tTGCAGTTTTTTTTTTTTTTT\t*",
    "tagSeq=F\t0\tChromosome_2\t500\t42\t25M\t*\t0\t0\tTGCAGACGTACGTACGTACGTACGT\t*",
    "tagSeq=G\t0\tChromosome_2\t500\t42\t20M\t*\t0\t0\tTGCAGACGTACGTACGTACG\t*",
    "tagSeq=H\t0\tChromosome_2\t500\t42\t25M\t*\t0\t0\tTGCAGACGTACGAACGTACGTACGT\t*",
    "tagSeq=I\t16\t3\t77\t42\t10M2D5M1I4M\t*\t0\t0\tAAACCCCGGGGTTTTCTGCA\t*",
    "tagSeq=J\t0\t3\t5\t42\t20M\t*\t0\t0\tTGCAGAAAACCCCGGGGTTA\t*",
    "tagSeq=K\t0\t3\t5\t42\t20M\t*\t0\t0\tTGCAGAAAACGCCGGGGTTA\t*",
    "tagSeq=L\t0\t3\t5\t42\t20M\t*\t0\t0\tTGCAGAATACCCCGGGGTTA\t*",
]) + "\n"

PYRAD = "\n".join([
    ">ind1_0     TGCAGAAAACCCCGGGGTTTT-",
    ">ind1_1     TGCAGAAAACCCCGGGGTTTT-",
    ">ind2_0     TGCAGAAAACCCTGGGGTTTT-",
    ">ind2_1     TGCAGAAAACCCTGGGGTTTTA",
    "//                      *         |1|",
    ">ind1_0     TGCAGCC-TTAACCGGTT",
    ">ind1_1     TGCAGCCATTAACCGGTT",
    ">ind2_0     TGCAGCCATTAACCNGTT",
    "//                 -           |2|",
    ">ind1_0     TGCAGGGGGGGGGGAAAA",
    "//                             |3|",
    ">ind1_0     TGCAGACACACACACACA",
    ">ind1_1     TGCAGACACATACACACA",
    ">ind2_1     TGCAGACACACACACGCA",
    "//                    *    *   |4*|",
]) + "\n"


def cases_readers():
    cases = []
    add = lambda func, files, *a, **kw: cases.append(
        run_case(func, files, a, kw.pop("kwargs", {}), kw.pop("outfiles", ())))
    # --- key file ---
    key = ("File,Barcode,Sample,Notes\nlane1.fq,AACG,s1,x\nlane1.fq, ttgca ,s2,y\n,,,\n"
           "lane2.fq.gz,AACG,s1,\nlane0.fq,GGT,s3,z\n")
    add("readBarcodeKeyfile", {"k.csv": key}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": key.replace("\n", "\r\n")}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "Sample,File,Barcode\ns1,a.fq,\ns2,b.fq,\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode\na.fq,ACGT\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode,Sample\na.fq,ACGT,\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode,Sample\n,ACGT,s\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode,Sample\na.fq,ACNT,s\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode,Sample\na.fq,ACGT,s\na.fq,acgt,t\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode,Sample\na.fq,ACGT\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "﻿File,Barcode,Sample\na.fq,ACGT,s\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": "File,Barcode,Sample\na.fq,,s\na.fq,,t\n"}, "k.csv")
    add("readBarcodeKeyfile", {"k.csv": 'File,Barcode,Sample\n"a,b.fq",ACGT,"s ""q"""\n'}, "k.csv")
    add("readBarcodeKeyfile", {}, "missing.csv")
    add("readBarcodeKeyfile", {"k.csv": "Input File,Barcode,Output File\na.fq,ACGT,o1.fq\na.fq,GG,o2.fq\n"},
        "k.csv", kwargs={"forSplitter": True})
    add("readBarcodeKeyfile", {"k.csv": "Input File,Barcode,Output File\na.fq,ACGT,o1.fq\nb.fq,GG,o1.fq\n"},
        "k.csv", kwargs={"forSplitter": True})
    add("readBarcodeKeyfile", {"k.csv": key}, "k.csv", kwargs={"forSplitter": True})
    # --- UNEAK ---
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK}, "t.fa")
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK}, "t.fa", kwargs={"toKeep": ["TP539"]})
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK}, "t.fa", kwargs={"toKeep": []})
    pad = (">TP1_query_20\nTGCAGACGTACGTACGTACGAAAAAAAAAA\n>TP1_hit_24\nTGCAGACGTACGTACGTTCGACGTAAAAAA\n"
           ">TP2_query_20\nTGCAGTTGTACGTACGTACGAAAAAAAAAA\n>TP2_hit_24\nTGCAGTTGTACGTACGTACGACGTAAAAAA\n"
           ">TP3_query_30\ntgcagcccccgtacgtacgtacgaaaaaaa\n>TP3_hit_30\nTGCAGCCCCCGTACGTACGAACGAAAAAAA\n")
    add("readTags_UNEAK_FASTA", {"t.fa": pad}, "t.fa")
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK + UNEAK[:160]}, "t.fa")          # duplicate sequence
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK.replace(">TP539_hit", ">TP540_hit")}, "t.fa")
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK.replace(">TP539_q", ">XX539_q")}, "t.fa")
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK.replace("GGTGCAT\n", "GGTGCNT\n", 1)}, "t.fa")
    add("readTags_UNEAK_FASTA", {"t.fa": UNEAK.replace("_64\n", "_x\n", 1)}, "t.fa")
    add("readTags_UNEAK_FASTA", {}, "missing.fa")
    # --- Merged ---
    add("readTags_Merged", {"t.csv": MERGED}, "t.csv")
    add("readTags_Merged", {"t.csv": MERGED}, "t.csv", kwargs={"toKeep": ["Mrkr2011", "TP276"]})
    dup = MERGED + "Dup1,TGCAGAAA[A/G]AAAAATCACAGCACAGGCACTAGAAGCACTGGTAGTAACTCGAGACAGGATGTAT,\n"
    add("readTags_Merged", {"t.csv": dup}, "t.csv")
    add("readTags_Merged", {"t.csv": dup}, "t.csv", kwargs={"allowDuplicates": True})
    add("readTags_Merged", {"t.csv": MERGED + "Bad_name,ACGT[A/C]TT,\n"}, "t.csv")
    add("readTags_Merged", {"t.csv": MERGED + "NoBr,ACGTACTT,\n"}, "t.csv")
    add("readTags_Merged", {"t.csv": MERGED + "BadSeq,ACGT[A/N]TT,\n"}, "t.csv")
    add("readTags_Merged", {"t.csv": MERGED + "\n"}, "t.csv")                   # blank trailing line
    add("readTags_Merged", {"t.csv": "Marker,Tag\nA,AC[G/T]\n"}, "t.csv")
    add("readTags_Merged", {"t.csv": "Tag sequence,Marker name\n ac[g/t]aa , m1 \n"}, "t.csv")
    add("readTags_Merged", {}, "missing.csv")
    # --- Columns ---
    add("readTags_Columns", {"t.csv": COLUMNS}, "t.csv")
    add("readTags_Columns", {"t.csv": COLUMNS}, "t.csv", kwargs={"toKeep": ["TP539"]})
    add("readTags_Columns", {"t.csv": COLUMNS + "M3,ACGTAC,AGGTAT,\nM4,ACGTAA,ACG,\n"}, "t.csv")
    add("readTags_Columns", {"t.csv": COLUMNS + "M_3,ACGTAC,AGGTAT,\n"}, "t.csv")
    add("readTags_Columns", {"t.csv": COLUMNS + "M3,ACGTNC,AGGTAT,\n"}, "t.csv")
    add("readTags_Columns", {"t.csv": COLUMNS + COLUMNS.split("\n")[1] + "\n"}, "t.csv")
    add("readTags_Columns", {"t.csv": "Marker name,Tag sequence 0\nA,AC\n"}, "t.csv")
    add("readTags_Columns", {"t.csv": COLUMNS + "\n"}, "t.csv")
    # --- Rows ---
    add("readTags_Rows", {"t.csv": ROWS}, "t.csv")
    add("readTags_Rows", {"t.csv": ROWS}, "t.csv", kwargs={"toKeep": ["Mrker4050"]})
    add("readTags_Rows", {"t.csv": ROWS + "M_1,0,ACGT,\n"}, "t.csv")
    add("readTags_Rows", {"t.csv": ROWS + "M1,0,ACXT,\n"}, "t.csv")
    add("readTags_Rows", {"t.csv": ROWS + "M9,0,AGTAGGGAAAGGCCGGTAAGGCAACTAAA,\n"}, "t.csv")
    add("readTags_Rows", {"t.csv": "Marker name,Allele,Tag sequence\nA,0,AC\n"}, "t.csv")
    add("readTags_Rows", {"t.csv": ROWS + "\n"}, "t.csv")
    add("readTags_Rows", {"t.csv": "Tag sequence,Allele name,Marker name\n acgt ,  x , m \n"}, "t.csv")
    # --- Stacks ---
    for ver in (1, 2):
        t, s, a = stacks_files(ver)
        files = {"c.tags.tsv": t, "c.snps.tsv": s, "c.alleles.tsv": a}
        for bo in (False, True):
            add("readTags_Stacks", files, "c.tags.tsv", "c.snps.tsv", "c.alleles.tsv",
                kwargs={"binaryOnly": bo, "version": ver})
        add("readTags_Stacks", files, "c.tags.tsv", "c.snps.tsv", "c.alleles.tsv",
            kwargs={"toKeep": ["1", "3"], "version": ver})
    t, s, a = stacks_files(1)
    gz = {"c.tags.tsv.gz": gzip.compress(t.encode()), "c.snps.tsv.gz": gzip.compress(s.encode()),
          "c.alleles.tsv.gz": gzip.compress(a.encode())}
    add("readTags_Stacks", gz, "c.tags.tsv.gz", "c.snps.tsv.gz", "c.alleles.tsv.gz")
    add("readTags_Stacks", {"c.tags.tsv": t, "c.snps.tsv": s, "c.alleles.tsv": a + "0\t1\t99\tA\t1\t1\n"},
        "c.tags.tsv", "c.snps.tsv", "c.alleles.tsv")
    add("readTags_Stacks", {"c.tags.tsv": t, "c.snps.tsv": "0\t1\t1\tx\n", "c.alleles.tsv": a},
        "c.tags.tsv", "c.snps.tsv", "c.alleles.tsv")
    add("readTags_Stacks", {"c.tags.tsv": "a\tb\n", "c.snps.tsv": s, "c.alleles.tsv": a},
        "c.tags.tsv", "c.snps.tsv", "c.alleles.tsv")
    add("readTags_Stacks", {}, "c.tags.tsv", "c.snps.tsv", "c.alleles.tsv")
    # --- TASSEL SAM ---
    add("readTags_TASSELSAM", {"t.sam": SAM}, "t.sam")
    add("readTags_TASSELSAM", {"t.sam": SAM}, "t.sam", kwargs={"binaryOnly": True})
    add("readTags_TASSELSAM", {"t.sam": SAM}, "t.sam", kwargs={"noMonomorphic": True})
    add("readTags_TASSELSAM", {"t.sam": SAM}, "t.sam", kwargs={"toKeep": ["S01_1012", "S3_15"]})
    add("readTags_TASSELSAM", {"t.sam": SAM}, "t.sam", kwargs={"toKeep": ["nothing"]})
    add("readTags_TASSELSAM", {"t.sam": SAM}, "t.sam",
        kwargs={"writeMarkerKey": True, "keyfilename": "key.csv", "binaryOnly": True},
        outfiles=["key.csv"])
    add("readTags_TASSELSAM", {"t.sam": SAM + "short\tline\n"}, "t.sam")
    add("readTags_TASSELSAM", {}, "missing.sam")
    # --- pyRAD ---
    add("readTags_pyRAD", {"t.alleles": PYRAD}, "t.alleles")
    add("readTags_pyRAD", {"t.alleles": PYRAD}, "t.alleles", kwargs={"binaryOnly": True})
    add("readTags_pyRAD", {"t.alleles": PYRAD}, "t.alleles", kwargs={"toKeep": ["2", "4"]})
    add("readTags_pyRAD", {"t.alleles": PYRAD + "garbage\n"}, "t.alleles")
    add("readTags_pyRAD", {"t.alleles": PYRAD.replace("ACACGCA", "ACACXCA")}, "t.alleles")
    add("readTags_pyRAD", {}, "missing.alleles")
    return cases


# ---------------------------------------------------------------------------
# 4. trim decision + splitter
# ---------------------------------------------------------------------------

def cases_trim():
    cases = []
    rng = random.Random(77)
    for aname in sorted(ref.adapters):
        adapter = ref.adapters[aname]
        cutsite = "TGCAG" if aname.startswith("PstI") else "TGCAT"
        barcodes = prefix_free_barcodes(rng, 5, cutsite, 4, 9)
        with contextlib.redirect_stdout(io.StringIO()):
            trees = ref.build_adapter_tree(adapter, barcodes)
        full0 = adapter[0][0].replace("^", "")
        full1 = adapter[1][0].replace("^", "")
        a0 = adapter[0][0][:adapter[0][0].find("^")] + adapter[0][1]
        seqs, barix, starts, slices = [], [], [], []
        for _ in range(160):
            bi = rng.randrange(len(barcodes))
            bc = barcodes[bi]
            a1 = adapter[1][0][:adapter[1][0].find("^")] + adapter[1][1].replace(
                "[barcode]", ref.reverseComplement(bc))
            insert = rand_seq(rng, rng.randint(0, 90))
            r = rng.random()
            if r < 0.30:
                tail = rng.choice([a0, a1])[:rng.randint(1, 70)]
            elif r < 0.40:
                tail = rng.choice([a0, a1]) + rand_seq(rng, rng.randint(1, 6))
            elif r < 0.55:
                tail = rng.choice([full0, full1]) + rand_seq(rng, rng.randint(0, 30))
            elif r < 0.62:
                tail = full0 + rand_seq(rng, 5) + full1 + rand_seq(rng, 4)
            elif r < 0.69:
                tail = full1 + rand_seq(rng, 5) + full0
            else:
                tail = rand_seq(rng, rng.randint(0, 40))
            s = (bc + cutsite + insert + tail)[:rng.choice([60, 100, 100, 150])]
            if rng.random() < 0.05:
                k = rng.randrange(len(s))
                s = s[:k] + "N" + s[k + 1:]
            start = len(bc) + len(cutsite)
            seqs.append(s)
            barix.append(bi)
            starts.append(start)
            slices.append(ref.findAdapterSeq(s, trees[bi], full0, full1, start))
        cases.append({"adapter_name": aname, "adapter": jsonable(adapter), "cutsite": cutsite,
                      "barcodes": barcodes, "indices": [t[1] for t in trees],
                      "seqs": seqs, "barindex": barix, "searchstart": starts, "slice2": slices})
    return cases


def cases_splitter():
    cases = []
    rng = random.Random(99)
    for aname, cutsite in (("PstI-MspI-Hall", "TGCAG"), ("NsiI-MspI-Clark", "TGCAT"),
                           ("PstI-MspI-Poland", "TGCAG")):
        adapter = ref.adapters[aname]
        barcodes = prefix_free_barcodes(rng, 4, cutsite, 4, 8)
        a0 = adapter[0][0][:adapter[0][0].find("^")] + adapter[0][1]
        reads = []
        for _ in range(120):
            bc = rng.choice(barcodes)
            ins = rand_seq(rng, rng.randint(5, 80))
            r = rng.random()
            if r < 0.4:
                s = bc + cutsite + ins + a0
            elif r < 0.6:
                s = bc + cutsite + ins + adapter[0][0].replace("^", "") + rand_seq(rng, 30)
            elif r < 0.8:
                s = bc + cutsite + ins + rand_seq(rng, 60)
            else:
                s = rand_seq(rng, 90)
            reads.append(s[:80])
        fq = fastq_text(rng, reads, newline=rng.choice(["\n", "\r\n"]), messy=True)
        outs = ["out%d.fq" % i for i in range(len(barcodes))]
        c = run_case("barcodeSplitter", {"in.fq": fq}, ("in.fq", barcodes, outs),
                     {"cutsite": cutsite, "adapter": adapter, "maxreads": 100}, outfiles=outs)
        c["stdout"] = ""
        cases.append(c)
    return cases


# ---------------------------------------------------------------------------
# 5. whole script runs (config-1 shape, reduced)
# ---------------------------------------------------------------------------

def pack_files(files):
    """File set -> JSON form.  FASTQ images are stored gzip+base64 ('gzb64')."""
    out = {}
    for name, content in files.items():
        if isinstance(content, bytes):
            out[name] = {"gzb64": base64.b64encode(gzip.compress(content, mtime=0)).decode()}
        else:
            out[name] = {"text": content}
    return out


def run_script(fileset, files, argv, outfiles):
    rec = {"fileset": fileset, "argv": argv}
    with tempfile.TemporaryDirectory() as tmp:
        for name, content in files.items():
            mode = "wb" if isinstance(content, bytes) else "w"
            with open(os.path.join(tmp, name), mode) as fh:
                fh.write(content)
        p = subprocess.run([sys.executable, "-W", "ignore", os.path.join(REF, "tagdigger_script.py")] + argv,
                           cwd=tmp, capture_output=True, text=True)
        rec["returncode"] = p.returncode
        rec["stderr_tail"] = p.stderr.strip().splitlines()[-1:] if p.stderr.strip() else []
        rec["outfiles"] = {}
        for name in outfiles:
            path = os.path.join(tmp, name)
            rec["outfiles"][name] = (base64.b64encode(open(path, "rb").read()).decode()
                                     if os.path.exists(path) else None)
    return rec


def cases_script():
    import numpy as np
    from tagdigger_b200 import synth
    cases = []
    rng = np.random.default_rng(20161)
    bcs = synth.make_barcodes(12, rng)
    names, alleles, seqs = synth.make_marker_pairs(40, rng)
    tags = [s for pair in seqs for s in pair]
    fq1, _ = synth.make_fastq(1500, bcs, tags, rng)
    fq2, _ = synth.make_fastq(900, bcs[:6], tags, rng, newline=b"\r\n")
    key = "File,Barcode,Sample\n"
    key += "".join("lane1.fq,%s,S%02d\n" % (b, i) for i, b in enumerate(bcs))
    key += "".join("lane2.fq.gz,%s,S%02d\n" % (b, (i * 5) % 12) for i, b in enumerate(bcs[:6]))
    files = {"lane1.fq": fq1, "lane2.fq.gz": gzip.compress(fq2), "key.csv": key,
             "tags.csv": synth.merged_csv(names, alleles, seqs),
             "keep.txt": "\n".join(names[::2]) + "\n"}
    cases.append(run_script("lanes", files, ["-e", "PstI", "--MergedTags", "tags.csv", "-b", "key.csv",
                                    "-o", "counts.csv", "-g", "geno.csv"], ["counts.csv", "geno.csv"]))
    cases.append(run_script("lanes", files, ["-c", "tgcag", "--MergedTags", "tags.csv", "-b", "key.csv",
                                    "-k", "keep.txt", "-o", "counts.csv"], ["counts.csv"]))
    # pre-split flow: blank barcodes
    pre = {}
    key2 = "File,Barcode,Sample\n"
    for i in range(3):
        fq, _ = synth.make_fastq(500, [""], tags, rng)
        pre["s%d.fq" % i] = fq
        key2 += "s%d.fq,,Sam%d\n" % (i, i % 2)
    pre["key.csv"] = key2
    pre["tags.csv"] = files["tags.csv"]
    cases.append(run_script("presplit", pre, ["-e", "PstI", "--MergedTags", "tags.csv", "-b", "key.csv",
                                  "-o", "counts.csv"], ["counts.csv"]))
    # argument errors
    cases.append(run_script("lanes", files, ["--MergedTags", "tags.csv", "-b", "key.csv", "-o", "c.csv"], ["c.csv"]))
    cases.append(run_script("lanes", files, ["-e", "PstI", "-c", "CWGC", "--MergedTags", "tags.csv", "-b", "key.csv",
                                    "-o", "c.csv"], ["c.csv"]))
    cases.append(run_script("lanes", files, ["-e", "PstI", "-b", "key.csv", "-o", "c.csv"], ["c.csv"]))
    return {"filesets": {"lanes": pack_files(files), "presplit": pack_files(pre)}, "cases": cases}



def cases_flow():
    """BASELINE config 5 as a flow, reduced: a two-enzyme (PstI-MspI) multiplexed library with adapter
    read-through is split by barcode and trimmed (barcode_splitter_script.py:8-36), the per-sample
    files are counted with a blank Barcode column and a marker-list filter (tagdigger_script.py -k).
    Both stages are run with the reference's own scripts; inputs, the split files and the final CSV
    are recorded."""
    import numpy as np
    from tagdigger_b200 import synth
    rng = np.random.default_rng(20165)
    bcs = synth.make_barcodes(8, rng)
    lens = rng.integers(30, 65, size=60)
    names, alleles, seqs = synth.make_marker_pairs(60, rng, lengths=lens)
    tags = [s for pair in seqs for s in pair]
    adapter = ref.adapters["PstI-MspI-Hall"]
    tail = (adapter[0][0].replace("^", "") + adapter[0][1]).encode()      # MspI remnant + common adapter
    fq, _ = synth.make_fastq(3000, bcs, tags, rng, adapter_tail=tail, p_nobarcode=0.10, p_unknown=0.25)
    split_key = "Input File,Barcode,Output File\n" + "".join("lib.fq,%s,sample%02d.fq\n" % (b, i) for i, b in enumerate(bcs))
    count_key = "File,Barcode,Sample\n" + "".join("sample%02d.fq,,S%02d\n" % (i, i % 6) for i in range(len(bcs)))
    files = {"lib.fq": fq, "split_key.csv": split_key, "count_key.csv": count_key,
             "tags.csv": synth.merged_csv(names, alleles, seqs), "keep.txt": "\n".join(names[::2]) + "\n"}
    rec = {"files": pack_files(files), "split_argv": ["-b", "split_key.csv", "-a", "PstI-MspI-Hall"],
           "count_argv": ["-e", "PstI", "--MergedTags", "tags.csv", "-k", "keep.txt", "-b", "count_key.csv", "-o", "counts.csv",
                          "-g", "geno.csv"]}
    with tempfile.TemporaryDirectory() as tmp:
        for name, content in files.items():
            with open(os.path.join(tmp, name), "wb" if isinstance(content, bytes) else "w") as fh:
                fh.write(content)
        p1 = subprocess.run([sys.executable, "-W", "ignore", os.path.join(REF, "barcode_splitter_script.py")] + rec["split_argv"],
                            cwd=tmp, capture_output=True, text=True)
        assert p1.returncode == 0, p1.stderr
        p2 = subprocess.run([sys.executable, "-W", "ignore", os.path.join(REF, "tagdigger_script.py")] + rec["count_argv"],
                            cwd=tmp, capture_output=True, text=True)
        assert p2.returncode == 0, p2.stderr
        import hashlib
        rec["split_sha256"] = {"sample%02d.fq" % i: hashlib.sha256(open(os.path.join(tmp, "sample%02d.fq" % i), "rb").read()).hexdigest()
                               for i in range(len(bcs))}                  # (the files themselves would triple the fixture)
        rec["outfiles"] = {n: base64.b64encode(open(os.path.join(tmp, n), "rb").read()).decode()
                           for n in ("counts.csv", "geno.csv")}
    return {"cases": [rec]}


def cases_find_tags_text():
    """Text-mode behaviour of find_tags_fastq's file reading (tagdigger_fun.py:240-243, 272-273):
    the file is decoded as UTF-8 (invalid bytes raise UnicodeDecodeError), and the loop stops at
    maxreads, so defects located after that point are never met."""
    cases = []

    def add(fq, barcodes, tags, name="a.fq", **kw):
        c = run_case("find_tags_fastq", {name: fq}, (name, barcodes, tags), kw)
        c["stdout"] = ""
        if len(fq) > 20000:               # the long filler compresses to nothing: keep the fixture small
            c["files"][name] = {"gzb64": base64.b64encode(gzip.compress(fq, mtime=0)).decode()}
        cases.append(c)

    one = lambda s, h="@h": (h + "\n%s\n+\n%s\n" % (s, "I" * len(s))).encode("utf-8")
    good = one("AACGTGCAGCCCC")
    add(good * 3, ["AACG"], ["CCCC"])
    add(one("AACGTGCAGCCCC", u"@h \u00e9\u20ac \U0001F9EC") * 3, ["AACG"], ["CCCC"])     # valid multi-byte text
    add(b"@h\xff\n" + good[3:] + good, ["AACG"], ["CCCC"])                            # invalid start byte
    add(good + b"@h\nAACG\xc3\x28TGCAGCCCC\n+\nIIII\n", ["AACG"], ["CCCC"])           # invalid continuation
    add(good + b"@h\nAACGTGCAGCCCC\n+\nIII\xed\xa0\x80\n", ["AACG"], ["CCCC"])        # surrogate
    add(good + b"@h\nAACGTGCAGCCCC\n+\nIII\xc0\xaf\n", ["AACG"], ["CCCC"])            # overlong form
    add(good * 2 + b"@h \xe2\x82", ["AACG"], ["CCCC"])                               # sequence cut by the end of the file
    add(good * 2 + b"@h \xf4\x90\x80\x80\n", ["AACG"], ["CCCC"])                      # above U+10FFFF
    filler = good * 3000                                                              # ~96 KB: several text-layer chunks
    add(good * 2 + filler + b"@h\xff\n" + good[3:], ["AACG"], ["CCCC"], maxreads=2)      # defect far behind the stop
    add(good * 2 + filler + b"@h\xff\n" + good[3:], ["AACG"], ["CCCC"])                  # the same file read to the end
    gz = gzip.compress(good * 2 + filler, mtime=0)
    add(gz[:len(gz) // 2], ["AACG"], ["CCCC"], name="cut.fq.gz", maxreads=2)           # truncated far behind the stop
    add(gz[:len(gz) // 2], ["AACG"], ["CCCC"], name="cut.fq.gz")
    add(gzip.compress(good * 2 + filler + b"@h\xff\n" + good[3:], mtime=0), ["AACG"], ["CCCC"], name="bad.fq.gz", maxreads=2)
    add(gzip.compress(good * 2 + b"@h\xff\n" + good[3:], mtime=0), ["AACG"], ["CCCC"], name="bad.fq.gz")
    return cases


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "text":          # only the cases added in round 2
        dump("find_tags_text.json", cases_find_tags_text())
        dump("flow.json", cases_flow())
        sys.exit(0)
    dump("find_tags.json", cases_find_tags())
    dump("small_functions.json", cases_small())
    dump("readers.json", cases_readers())
    dump("trim.json", cases_trim())
    dump("splitter.json", cases_splitter())
    dump("script.json", cases_script())
    dump("find_tags_text.json", cases_find_tags_text())
    dump("flow.json", cases_flow())
