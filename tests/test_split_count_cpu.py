"""Counting adapter-trimmed reads in one pass (count_files(..., adapter=...), tagdigger_script
--adapter): the oracle's two-stage composition against the recorded two-stage run of the reference,
and the checks that come before any GPU work."""

import base64
import contextlib
import io
import os

import pytest

from conftest import load_golden, materialize
from oracle import tagdigger_oracle as orc
from split_count_check import two_stage
from tagdigger_b200 import counting, hostio, tagdigger_script

FLOW = load_golden("flow.json")["cases"][0]


def flow_inputs(directory):
    """The recorded flow as a one-pass run: the library, its File,Barcode,Sample key (barcode ->
    sample through the split key and the count key) and the kept, sanitised tags."""
    materialize(FLOW["files"], directory)
    split = hostio.readBarcodeKeyfile(os.path.join(str(directory), "split_key.csv"), forSplitter=True)
    count = hostio.readBarcodeKeyfile(os.path.join(str(directory), "count_key.csv"))
    (lib, (barcodes, outputs)), = split.items()
    key = {lib: [list(barcodes), [count[o][1][0] for o in outputs]]}
    keep = hostio.readMarkerNames(os.path.join(str(directory), "keep.txt"))
    names, seqs = hostio.sanitizeTags(hostio.readTags_Merged(os.path.join(str(directory), "tags.csv"), toKeep=keep))
    return lib, key, names, seqs


def test_oracle_two_stage_reproduces_the_recorded_flow(tmp_path):
    lib, key, names, seqs = flow_inputs(tmp_path)
    with open(os.path.join(str(tmp_path), lib), "rb") as fh:
        text = fh.read().decode("utf-8")
    with contextlib.redirect_stdout(io.StringIO()):
        samples, counts, totals = two_stage({lib: text}, key, seqs, "TGCAG", hostio.adapters["PstI-MspI-Hall"], "TGCAG")
    want = base64.b64decode(FLOW["outfiles"]["counts.csv"])
    assert orc.counts_csv_bytes(counts, samples, names) == want
    assert len(want) == 1489
    reads, bar, clipped, hits = totals[lib]
    assert reads > bar > clipped > 0 and hits == sum(map(sum, counts))


def test_cli_adapter_option():
    p = tagdigger_script.build_parser()
    base = ["-e", "PstI", "--MergedTags", "t.csv", "-b", "k.csv", "-o", "o.csv"]
    assert p.parse_args(base).adapter is None
    for name in sorted(hostio.adapters):
        assert p.parse_args(base + ["--adapter", name]).adapter == name
    with pytest.raises(SystemExit):
        p.parse_args(base + ["--adapter", "PstI-MspI-Nobody"])


KEY = {"lib.fq": [["ACGTA", "TTGCAC"], ["S1", "S2"]]}
TAGS = ["TGCAGACGTTAGC", "TGCAGACGTTAGA"]


@pytest.mark.parametrize("kwargs, error, match", [
    (dict(maxreads=1000), ValueError, "maxreads"),
    (dict(split_maxreads=5e9 + 1), ValueError, "split_maxreads"),
    (dict(split_maxreads=None), ValueError, "split_maxreads"),
    (dict(adapter="PstI-MspI-Nobody"), ValueError, "unknown adapter set"),
    (dict(split_cutsite="TGCAN"), AssertionError, "Only ACGT cut sites allowed."),
    (dict(key={"lib.fq": [["ACGTA", "TTGNAC"], ["S1", "S2"]]}), AssertionError, "Found non-ACGT barcodes."),
    (dict(key={"lib.fq": [["ACTGCAGA", "AC"], ["S1", "S2"]]}), AssertionError, "Problematic sequence: 1"),
    (dict(tags=["TGCAGACGXTAGC"]), AssertionError, "Non-ACGT tag."),
    (dict(tags=[]), IndexError, "list index out of range"),
])
def test_set_up_errors_come_before_any_gpu_work(kwargs, error, match):
    args = dict(key=KEY, tags=TAGS, adapter="PstI-MspI-Hall")
    args.update(kwargs)
    key, tags = args.pop("key"), args.pop("tags")
    with pytest.raises(error, match=match):
        counting.count_files(key, tags, "TGCAG", **args)
