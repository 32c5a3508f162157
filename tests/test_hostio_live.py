"""Live differential fuzzing of the host API mirror against the reference (skipped where the
reference is not staged in oracle/_ref).  Every recorded reader case is re-run on randomly
damaged copies of its input files -- lines dropped, duplicated, swapped, characters substituted --
and the mirror must agree with the reference on return value, printed messages and exception."""

import contextlib
import io
import random

import pytest

from conftest import NO_REFERENCE, file_bytes, have_reference, import_reference, load_golden
from tagdigger_b200 import hostio

pytestmark = pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)

READERS = load_golden("readers.json")


def _mutate(rng, text):
    lines = text.split("\n")
    for _ in range(rng.randint(1, 3)):
        if not lines:
            break
        k = rng.random()
        i = rng.randrange(len(lines))
        if k < 0.2:
            del lines[i]
        elif k < 0.4:
            lines.insert(i, lines[i])
        elif k < 0.55 and len(lines) > 1:
            j = rng.randrange(len(lines))
            lines[i], lines[j] = lines[j], lines[i]
        elif lines[i]:
            p = rng.randrange(len(lines[i]))
            c = rng.choice("ACGTN_-[]/,\t >0123456789acgtXx|*")
            lines[i] = lines[i][:p] + c + lines[i][p + (0 if rng.random() < 0.3 else 1):]
    return "\n".join(lines)


def _run(fn, args, kwargs):
    out = io.StringIO()
    ret, exc = None, None
    with contextlib.redirect_stdout(out):
        try:
            ret = fn(*args, **kwargs)
        except BaseException as e:  # noqa: BLE001
            exc = (type(e).__name__, str(e))
    return ret, exc, out.getvalue()


@pytest.mark.parametrize("i", range(len(READERS)))
def test_reader_fuzz_live(i, in_tmp):
    ref = import_reference()
    case = READERS[i]
    rng = random.Random(4242 + i)
    texts = {}
    for name, spec in case["files"].items():
        try:
            texts[name] = file_bytes(spec).decode("utf-8")
        except UnicodeDecodeError:
            return
    for trial in range(60):
        for name, text in texts.items():
            if name.endswith(".gz"):
                continue
            with open(name, "w", newline="") as fh:
                fh.write(_mutate(rng, text) if trial else text)
        kwargs = dict(case["kwargs"])
        want = _run(getattr(ref, case["func"]), case["args"], kwargs)
        got = _run(getattr(hostio, case["func"]), case["args"], dict(case["kwargs"]))
        assert got == want, (case["func"], trial)


def _rand_seq(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


@pytest.mark.parametrize("seed", range(40))
def test_sanitize_merge_write_live(seed, in_tmp):
    """sanitizeTags, extractMarkers, combineReadCounts, writeCounts, writeDiploidGeno on random
    inputs built to trigger the quirks (prefix overlaps, marker-name prefixes, equal sample names,
    markers without allele 0/1, names that need CSV quoting)."""
    ref = import_reference()
    rng = random.Random(900 + seed)
    names, seqs = [], []
    for m in range(rng.randint(1, 14)):
        marker = rng.choice(["TP%d" % rng.randint(1, 20), "M%d" % m, "x,y%d" % m, 'q"%d' % m, "L-%d" % m])
        base = "TGCAG" + _rand_seq(rng, rng.randint(3, 12))
        for a in range(rng.choice([1, 2, 2, 2, 3])):
            s = base if rng.random() < 0.15 else base[:rng.randint(4, len(base))] + _rand_seq(rng, rng.randint(0, 5))
            names.append("%s_%s_%s" % (marker, rng.choice("ACGT"), a) if rng.random() < 0.9 else marker + str(a))
            seqs.append(s)
    a = _run(ref.sanitizeTags, ([list(names), list(seqs)],), {})
    b = _run(hostio.sanitizeTags, ([list(names), list(seqs)],), {})
    assert a == b
    a = _run(ref.extractMarkers, (list(names),), {})
    b = _run(hostio.extractMarkers, (list(names),), {})
    assert a == b
    if a[1] is not None or not names:
        return
    ncol = len(names)
    files = ["f%d.fq" % k for k in range(rng.randint(1, 4))]
    bckeys, counts = {}, {}
    for f in files:
        nb = rng.randint(1, 4)
        bckeys[f] = [[_rand_seq(rng, 4) for _ in range(nb)], [rng.choice(["s1", "s2", "s,3", "s4 ", ""]) + str(rng.randint(0, 2)) for _ in range(nb)]]
        counts[f] = [[rng.choice([0, 0, 1, 5, 1000000]) for _ in range(ncol)] for _ in range(nb)]
    ca = _run(ref.combineReadCounts, ({f: [list(r) for r in counts[f]] for f in files}, bckeys), {})
    cb = _run(hostio.combineReadCounts, ({f: [list(r) for r in counts[f]] for f in files}, bckeys), {})
    assert ca == cb
    samples, matrix = ca[0]
    for fn in ("writeCounts", "writeDiploidGeno"):
        ra = _run(getattr(ref, fn), ("ref.csv", matrix, samples, list(names)), {})
        rb = _run(getattr(hostio, fn), ("mine.csv", matrix, samples, list(names)), {})
        assert ra == rb, fn
        import os
        assert os.path.exists("ref.csv") == os.path.exists("mine.csv")
        if os.path.exists("ref.csv"):
            assert open("ref.csv", "rb").read() == open("mine.csv", "rb").read(), fn
            os.remove("ref.csv")
            os.remove("mine.csv")
