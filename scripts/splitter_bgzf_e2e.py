#!/usr/bin/env python3
"""The barcode splitter with plain and with BGZF output files, on the config-5 shape (PstI-MspI-Hall
adapters, 96-plex, 150 bp reads with adapter read-through; scripts/config5_flow.py): the two runs
alternate, twice each.  Reported: split reads/s of each; the device time of the BGZF kernels
(deflate, scan, pack; CUDA events) and GB/s of uncompressed input through them; the compressed /
plain ratio; zlib level 1 over the same 65,280-byte members on every host thread, the alternative a
user has today; the card's name and power limit.

    python scripts/splitter_bgzf_e2e.py [reads] [out.json]
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
import zlib
from concurrent.futures import ThreadPoolExecutor

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))
import numpy as np  # noqa: E402

BLOCK = 65280


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, universal_newlines=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown (%s)" % e}


def zlib1_members(files, threads):
    """zlib level 1 over the 65,280-byte cuts of every file, one member per task: (seconds, bytes)."""
    jobs = []
    for f in files:
        with open(f, "rb") as fh:
            d = fh.read()
        jobs += [d[k:k + BLOCK] for k in range(0, len(d), BLOCK)]

    def one(b):
        c = zlib.compressobj(1, zlib.DEFLATED, -15)
        return len(c.compress(b) + c.flush()) + 26

    with ThreadPoolExecutor(max_workers=threads) as pool:
        t0 = time.perf_counter()
        sizes = list(pool.map(one, jobs, chunksize=16))
        t1 = time.perf_counter()
    return t1 - t0, sum(sizes) + 28 * len(files)


def main():
    import config5_flow
    from tagdigger_b200 import counting, hostio, splitter, synth
    reads = int(sys.argv[1]) if len(sys.argv) > 1 else 8_000_000
    out_json = sys.argv[2] if len(sys.argv) > 2 else None
    rng = random.Random(5)
    nrng = np.random.default_rng(5)
    adapter = hostio.adapters["PstI-MspI-Hall"]
    barcodes = synth.make_barcodes(96, nrng)
    _, _, seqs = synth.make_marker_pairs(2000, nrng)
    tags = [s for p in seqs for s in p]
    unit = min(reads, 250_000)
    text = config5_flow.make_reads(rng, barcodes, tags, adapter, unit)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    tmp = tempfile.mkdtemp(prefix="tdg_bgzf_", dir=os.environ.get("TDG_TMP", base))
    inp = os.path.join(tmp, "reads.fastq")
    with open(inp, "w") as fh:
        for _ in range(max(1, reads // unit)):
            fh.write(text)
    reads = max(1, reads // unit) * unit
    plain = [os.path.join(tmp, "s%02d.fq" % i) for i in range(len(barcodes))]
    comp = [os.path.join(tmp, "s%02d.fq.gz" % i) for i in range(len(barcodes))]
    eng = counting.get_engine(0)
    res = {"config": "config-5 shape: %d reads (150 bp), PstI-MspI-Hall adapters, 96-plex" % reads, "reads": reads,
           "input_MB": round(os.path.getsize(inp) / 1e6, 1), "host_cpus": os.cpu_count(), **card(), "runs": []}
    with contextlib.redirect_stdout(io.StringIO()):                 # warm-up: module load, buffers, both paths
        splitter.barcodeSplitter(inp, barcodes, plain, adapter=adapter, maxreads=300000)
        splitter.barcodeSplitter(inp, barcodes, comp, adapter=adapter, maxreads=300000, bgzf=True)
    for rep in range(2):
        for bgzf, outs in ((False, plain), (True, comp)):
            for o in outs:
                if os.path.exists(o):
                    os.remove(o)
            eng.timing_begin()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                splitter.barcodeSplitter(inp, barcodes, outs, adapter=adapter, bgzf=bgzf)
            t1 = time.perf_counter()
            ms, n = eng.timing_end()
            run = {"bgzf": bgzf, "split_s": round(t1 - t0, 3), "split_reads_per_s": round(reads / (t1 - t0), 1)}
            if bgzf:
                run["bgzf_kernel_ms"] = round(ms, 2)
                run["bgzf_kernel_sequences"] = n
            res["runs"].append(run)
    plain_bytes = sum(os.path.getsize(o) for o in plain)
    comp_bytes = sum(os.path.getsize(o) for o in comp)
    ok = True
    for p, z in zip(plain[:3], comp[:3]):
        import gzip
        with open(p, "rb") as a, open(z, "rb") as b:
            ok &= gzip.decompress(b.read()) == a.read()
    kms = [r["bgzf_kernel_ms"] for r in res["runs"] if r["bgzf"]]
    res["plain_output_MB"] = round(plain_bytes / 1e6, 1)
    res["bgzf_output_MB"] = round(comp_bytes / 1e6, 1)
    res["ratio_bgzf_to_plain"] = round(comp_bytes / plain_bytes, 4)
    res["bgzf_kernels_GB_per_s_of_input"] = round(plain_bytes / (min(kms) / 1e3) / 1e9, 2)
    zs, zbytes = zlib1_members(plain, os.cpu_count())
    res["zlib1_host"] = {"threads": os.cpu_count(), "s": round(zs, 3), "GB_per_s": round(plain_bytes / zs / 1e9, 3),
                         "ratio_to_plain": round(zbytes / plain_bytes, 4)}
    res["bgzf_size_vs_zlib1"] = round(comp_bytes / zbytes, 4)
    sp = [r["split_reads_per_s"] for r in res["runs"] if not r["bgzf"]]
    sz = [r["split_reads_per_s"] for r in res["runs"] if r["bgzf"]]
    res["bgzf_split_vs_plain_split"] = round(max(sz) / max(sp), 3)
    res["first_files_inflate_to_plain"] = "ok (3 samples)" if ok else "FAILED"
    print(json.dumps(res))
    if out_json:
        os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
        with open(out_json, "w") as fh:
            json.dump(res, fh, indent=1)
    for p in plain + comp + [inp]:
        if os.path.exists(p):
            os.remove(p)
    os.rmdir(tmp)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
