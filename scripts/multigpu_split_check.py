#!/usr/bin/env python3
"""Run on a box with >= 2 GPUs: barcode_splitter_script under torchrun at world N, on one library file
(plain FASTQ with LF and with CRLF line ends, and BGZF), splits that file on every rank at once.  Every
output file must have the md5 of the single-process run's, and rank 0's output must equal that run's.

    python scripts/multigpu_split_check.py 2
"""
import hashlib
import os
import random
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))
sys.path.insert(0, os.path.join(REPO, "tests"))
from multigpu_check import rank0_stdout  # noqa: E402


def library(reads):
    import numpy as np
    import config5_flow
    from tagdigger_b200 import hostio, synth
    nrng = np.random.default_rng(7)
    barcodes = synth.make_barcodes(24, nrng)
    _, _, seqs = synth.make_marker_pairs(300, nrng)
    text = config5_flow.make_reads(random.Random(7), barcodes, [s for p in seqs for s in p],
                                   hostio.adapters["PstI-MspI-Hall"], reads)
    return barcodes, text


def md5s(paths):
    return [hashlib.md5(open(p, "rb").read()).hexdigest() if os.path.exists(p) else None for p in paths]


def one_case(n, barcodes, name, data, port):
    from feed_check import bgzf_compress
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, name), "wb") as fh:
            fh.write(bgzf_compress(data) if name.endswith(".gz") else data)
        sums, stdout = {}, {}
        for world in (1, n):
            os.makedirs(os.path.join(tmp, "w%d" % world))
            outs = [os.path.join("w%d" % world, "s%02d.fq" % i) for i in range(len(barcodes))]
            with open(os.path.join(tmp, "key%d.csv" % world), "w") as fh:
                fh.write("Input File,Barcode,Output File\n" + "".join("%s,%s,%s\n" % (name, b, o) for b, o in zip(barcodes, outs)))
            argv = ["-b", "key%d.csv" % world, "-a", "PstI-MspI-Hall"]
            env = dict(os.environ, PYTHONPATH=REPO)
            if world == 1:
                cmd = [sys.executable, "-m", "tagdigger_b200.barcode_splitter_script"] + argv
            else:
                cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                       "--master-addr", "127.0.0.1", "--master-port", str(port),
                       "--log-dir", os.path.join(tmp, "logs"), "--redirects", "1",        # every rank's stdout to a file
                       "-m", "tagdigger_b200.barcode_splitter_script"] + argv
            p = subprocess.run(cmd, cwd=tmp, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, universal_newlines=True)
            sums[world] = md5s([os.path.join(tmp, o) for o in outs]) if p.returncode == 0 else None
            stdout[world] = p.stdout if world == 1 else rank0_stdout(os.path.join(tmp, "logs"))
            if p.returncode != 0:
                print(p.stdout[-2000:] + p.stderr[-2000:])
        ok = sums[1] is not None and None not in sums[1] and sums[1] == sums[n] and stdout[1] == stdout[n]
        print("world=%d one library file (%s) split on every rank: %s" % (n, name, "OK" if ok else "MISMATCH"))
        if ok:
            print("  md5 of %d output files equal; first: %s" % (len(sums[1]), sums[1][0]))
        return 0 if ok else 1


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 2
    barcodes, text = library(120000)
    data = text.encode("utf-8")
    bad = 0
    bad += one_case(n, barcodes, "lane.fq", data, 29541)
    bad += one_case(n, barcodes, "lane_crlf.fq", data.replace(b"\n", b"\r\n"), 29542)
    bad += one_case(n, barcodes, "lane.fq.gz", data, 29543)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
