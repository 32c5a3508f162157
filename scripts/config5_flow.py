#!/usr/bin/env python3
"""BASELINE config 5 as a flow, timed: a PstI-MspI library with adapter read-through (96-plex) is split
by barcode and trimmed (splitter.barcodeSplitter: /root/reference/barcode_splitter_script.py:8-36 ->
tagdigger_fun.py:1286-1368), then the 96 per-sample files are counted with a blank Barcode column
against the markers a keep-list leaves (tagdigger_script.py -k: :71-76, :123-133) --
counting.count_files.  Reported: reads/s of each stage and of the flow; checked: the count rows of the
first samples against the C oracle run over the split files, cell by cell.

The fused leg counts the same library in one pass (count_files(..., adapter=...): split, trim and count
on the GPU without the split files), alternating with the two-stage flow in the same process; its matrix
must equal the two-stage matrix in every cell.  Reported for it: reads/s, the device time of its blocks
(CUDA events around every block's upload and kernels), the time the host feed alone takes to read the
input, and the GPU's name and power limit.

    python scripts/config5_flow.py [reads]
"""
import contextlib
import io
import json
import os
import random
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402


def make_reads(rng, barcodes, tags, adapter, n):
    from tagdigger_b200 import hostio
    full0 = adapter[0][0].replace("^", "")
    rc = {bc: hostio.reverseComplement(bc) for bc in barcodes}
    out = []
    for i in range(n):
        bc = barcodes[rng.randrange(len(barcodes))]
        a1 = adapter[1][0][:adapter[1][0].find("^")] + adapter[1][1].replace("[barcode]", rc[bc])
        k = rng.random()
        body = tags[rng.randrange(len(tags))] if rng.random() < 0.6 else "TGCAG" + "".join(rng.choices("ACGT", k=59))
        insert = body + "".join(rng.choices("ACGT", k=rng.randint(0, 60)))
        if k < 0.35:
            tail = a1 + "".join(rng.choices("ACGT", k=40))                    # read-through into the adapter
        elif k < 0.38:
            tail = full0 + "".join(rng.choices("ACGT", k=60))                  # chimera
        else:
            tail = "".join(rng.choices("ACGT", k=100))
        head = bc if rng.random() < 0.9 else "".join(rng.choices("ACGT", k=6))
        s = (head + insert + tail)[:150]
        q = "".join(rng.choices("ABCDEFGHIJ", k=len(s)))
        out.append("@INST:7:FC:1:%d:%d:%d 1:N:0:ATCACG\n%s\n+\n%s\n" % (1100 + i % 90, rng.randrange(30000), rng.randrange(30000), s, q))
    return "".join(out)


def gpu_name_and_power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, universal_newlines=True, timeout=60).stdout
        return out.splitlines()[0].strip()
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def feed_seconds(_native, path):
    """The host feed alone (splitter.BLOCK_BYTES per read, into pinned memory): what the fused pass reads through."""
    from tagdigger_b200 import counting, splitter
    eng = counting.get_engine()
    buf = eng.host_alloc(splitter.BLOCK_BYTES)
    feed = _native.Feed(path, False)
    t0 = time.perf_counter()
    while feed.read_into(buf, splitter.BLOCK_BYTES):
        pass
    t1 = time.perf_counter()
    feed.close()
    eng.host_free(buf)
    return t1 - t0


def main():
    from oracle import c_oracle
    from tagdigger_b200 import _native, counting, hostio, splitter, synth
    reads = int(sys.argv[1]) if len(sys.argv) > 1 else 8_000_000
    rng = random.Random(5)
    nrng = np.random.default_rng(5)
    adapter = hostio.adapters["PstI-MspI-Hall"]
    barcodes = synth.make_barcodes(96, nrng)
    names, _, seqs = synth.make_marker_pairs(2000, nrng)
    tags = [s for p in seqs for s in p]
    keep = set(names[::2])                                    # the marker list keeps every second marker
    kept_tags = [s for name, p in zip(names, seqs) if name in keep for s in p]
    unit = 250_000
    text = make_reads(rng, barcodes, tags, adapter, unit)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    tmp = tempfile.mkdtemp(prefix="tdg_c5_", dir=os.environ.get("TDG_TMP", base))
    inp = os.path.join(tmp, "reads.fastq")
    with open(inp, "w") as fh:
        for _ in range(max(1, reads // unit)):
            fh.write(text)
    reads = max(1, reads // unit) * unit
    outs = [os.path.join(tmp, "s%02d.fq" % i) for i in range(len(barcodes))]
    bckeys = {outs[i]: [[""], ["Sample%02d" % i]] for i in range(len(barcodes))}
    res = {"config": "configs[4] as a flow: %d reads (150 bp), PstI-MspI-Hall adapters, 96-plex, %d tags of which a marker list keeps %d"
                     % (reads, len(tags), len(kept_tags)),
           "reads": reads, "input_MB": round(os.path.getsize(inp) / 1e6, 1), "host_cpus": os.cpu_count(), "runs": []}
    fused_key = {inp: [list(barcodes), ["Sample%02d" % i for i in range(len(barcodes))]]}
    res["gpu"] = gpu_name_and_power_limit()
    res["feed_s"] = round(feed_seconds(_native, inp), 3)
    res["fused_runs"] = []
    counts = None
    same = True
    for rep in range(3):
        for o in outs:
            if os.path.exists(o):
                os.remove(o)
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            splitter.barcodeSplitter(inp, barcodes, outs, adapter=adapter)
        t1 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            samples, counts = counting.count_files(bckeys, kept_tags, "TGCAG", as_array=True)
        t2 = time.perf_counter()
        res["runs"].append({"split_s": round(t1 - t0, 3), "count_s": round(t2 - t1, 3),
                            "split_reads_per_s": round(reads / (t1 - t0), 1), "count_reads_per_s": round(reads / (t2 - t1), 1),
                            "flow_reads_per_s": round(reads / (t2 - t0), 1)})
        eng = counting.get_engine()
        t0 = time.perf_counter()
        eng.timing_begin()
        with contextlib.redirect_stdout(io.StringIO()):
            _, fused = counting.count_files(fused_key, kept_tags, "TGCAG", as_array=True, adapter="PstI-MspI-Hall")
        ms, blocks = eng.timing_end()
        t1 = time.perf_counter()
        same &= bool(np.array_equal(fused, counts))
        res["fused_runs"].append({"fused_s": round(t1 - t0, 3), "fused_reads_per_s": round(reads / (t1 - t0), 1),
                                  "block_device_ms": round(ms, 1), "blocks": blocks})
    res["split_output_MB"] = round(sum(os.path.getsize(o) for o in outs) / 1e6, 1)
    res["tag_hits"] = int(np.asarray(counts).sum())
    ok = True
    for i in (0, 1, 95):
        with open(outs[i], "rb") as fh:
            want, _ = c_oracle.Counter([""], kept_tags, "TGCAG").count(fh.read())
        ok &= bool((np.asarray(counts[i]) == want[0]).all())
    res["rows_equal_c_oracle_on_split_files"] = "ok (3 samples)" if ok else "FAILED"
    res["fused_matrix_equals_two_stage"] = "ok (every cell)" if same else "FAILED"
    ok &= same
    print(json.dumps(res))
    for p in outs + [inp]:
        os.remove(p)
    os.rmdir(tmp)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
