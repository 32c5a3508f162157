"""The two-stage run that count_files(..., adapter=...) stands for, composed from the oracle:
barcodeSplitter's records (orc.split_records) -> one text per barcode -> find_tags_text(text, [''],
tags, cutsite) -> rows merged by sample (orc.combine_read_counts).  And reads of a PstI/NsiI-MspI
library that run into the adapter, for the tests that hold the GPU's one-pass count to it."""

import io

from helpers import rand_seq
from oracle import tagdigger_oracle as orc
from tagdigger_b200 import hostio


def two_stage(texts, key, tags, cutsite, adapter, split_cutsite, split_maxreads=500000000):
    """texts: {file: decoded text}; key: {file: [barcodes, samples]} (readBarcodeKeyfile's form).
    Returns (samples, counts, totals) with totals[file] = [reads, with barcode and cut site, clipped
    on the 3' end, with tag]."""
    per_output, out_key, totals = {}, {}, {}
    for f in sorted(key):
        barcodes, samples = key[f]
        bufs = [io.StringIO() for _ in barcodes]
        reads = bar = clipped = hits = 0
        for b, lines, s2 in orc.split_records(io.StringIO(texts[f], newline=None), barcodes, split_cutsite, adapter,
                                              split_maxreads, every=True):
            reads += 1
            if b > -1:
                bar += 1
                clipped += s2 != 999
                bufs[b].write("".join(ln + "\n" for ln in lines))
        for i, buf in enumerate(bufs):
            tot = []
            per_output[(f, i)] = orc.find_tags_text(buf.getvalue().encode("utf-8"), [""], tags, cutsite, totals=tot)
            out_key[(f, i)] = [[""], [samples[i]]]
            hits += tot[2]
        totals[f] = [reads, bar, clipped, hits]
    samples, counts = orc.combine_read_counts(per_output, out_key)
    return samples, counts, totals


def make_tags(rng, site, n):
    """n distinct tags that start with the cut site (about one in six holds MspI's CCGG)."""
    tags = set()
    while len(tags) < n:
        tags.add(site + rand_seq(rng, rng.randint(30, 60)))
    return sorted(tags)


def make_reads(rng, barcodes, site, tags, adapter, n, newline="\n"):
    """Reads of barcode + cut site + insert, many of them running into the common-cutter site or the
    adapter; some without a known barcode, some with N, lower case or blanks around the sequence."""
    full0 = adapter[0][0].replace("^", "")
    a0 = adapter[0][0][:adapter[0][0].find("^")] + adapter[0][1]
    out = []
    for i in range(n):
        bc = rng.choice(barcodes)
        a1 = adapter[1][0][:adapter[1][0].find("^")] + adapter[1][1].replace("[barcode]", hostio.reverseComplement(bc))
        body = rng.choice(tags) if rng.random() < 0.7 else site + rand_seq(rng, 50)
        insert = body[:rng.randint(len(body) - 10, len(body))] if rng.random() < 0.2 else body
        k = rng.random()
        if k < 0.3:
            tail = rng.choice([a0, a1])[:rng.randint(1, 70)]
        elif k < 0.45:
            tail = full0 + rand_seq(rng, rng.randint(0, 30))
        else:
            tail = rand_seq(rng, rng.randint(0, 80))
        head = bc if rng.random() < 0.9 else rand_seq(rng, rng.randint(0, 8))
        s = (head + insert + tail)[:rng.choice([60, 100, 150, 150])]
        w = rng.random()
        if s and w < 0.05:
            j = rng.randrange(len(s))
            s = s[:j] + "N" + s[j + 1:]
        elif w < 0.1:
            s = s.lower()
        elif w < 0.13:
            s = " " + s + "\t "
        q = "".join(rng.choice("ABCDEFGHIJ#") for _ in range(len(s.strip())))
        c2 = "+" if rng.random() < 0.8 else "+r%d" % i
        out.append("@r%d 1:N:0%s%s%s%s%s%s%s" % (i, newline, s, newline, c2, newline, q, newline))
    return "".join(out)
