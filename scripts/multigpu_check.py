#!/usr/bin/env python3
"""Run on a box with >= 2 GPUs: the golden 'lanes' script case under torchrun
(files dealt to the ranks, one NCCL all-reduce) must give the byte-identical CSVs.

    python scripts/multigpu_check.py 2
"""
import base64
import json
import os
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "tests"))
sys.path.insert(0, REPO)
from conftest import file_bytes  # noqa: E402


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 2
    gold = json.load(open(os.path.join(REPO, "tests", "golden", "script.json")))
    bad = 0
    for case in gold["cases"]:
        if case["returncode"] != 0:
            continue
        with tempfile.TemporaryDirectory() as tmp:
            for name, spec in gold["filesets"][case["fileset"]].items():
                with open(os.path.join(tmp, name), "wb") as fh:
                    fh.write(file_bytes(spec))
            env = dict(os.environ, PYTHONPATH=REPO)
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                   "--master-addr", "127.0.0.1", "--master-port", "29533", "-m", "tagdigger_b200.tagdigger_script"] + case["argv"]
            p = subprocess.run(cmd, cwd=tmp, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, universal_newlines=True)
            ok = p.returncode == 0
            for name, b64 in case["outfiles"].items():
                path = os.path.join(tmp, name)
                ok = ok and os.path.exists(path) and open(path, "rb").read() == base64.b64decode(b64)
            print("world=%d %s %s" % (n, " ".join(case["argv"]), "OK" if ok else "MISMATCH"))
            if not ok:
                bad += 1
                print(p.stdout[-3000:])
    bad += sharded_single_file(n)
    return 1 if bad else 0


def sharded_single_file(n):
    """One plain FASTQ file, fewer files than ranks: the file is cut into byte ranges, each rank
    counts the lines of its range, the counts are exchanged, and the result must equal the
    single-rank run and the C oracle -- with LF and with CRLF line ends, and with maxreads-free
    counting of a file whose ranges start mid-record.  Rank 0's output must equal the single-rank
    run's."""
    import numpy as np
    from oracle import c_oracle
    from tagdigger_b200 import synth
    rng = np.random.default_rng(99)
    bcs = synth.make_barcodes(10, rng)
    names, alleles, seqs = synth.make_marker_pairs(50, rng)
    tags = [s for p in seqs for s in p]
    bad = 0
    for newline in (b"\n", b"\r\n"):
        fq, _ = synth.make_fastq(60000, bcs, tags, rng, newline=newline)
        with tempfile.TemporaryDirectory() as tmp:
            open(os.path.join(tmp, "big.fq"), "wb").write(fq)
            open(os.path.join(tmp, "tags.csv"), "w").write(synth.merged_csv(names, alleles, seqs))
            open(os.path.join(tmp, "key.csv"), "w").write("File,Barcode,Sample\n" + "".join(
                "big.fq,%s,S%02d\n" % (b, i) for i, b in enumerate(bcs)))
            outs, stdout = {}, {}
            for world in (1, n):
                env = dict(os.environ, PYTHONPATH=REPO)
                argv = ["-e", "PstI", "--MergedTags", "tags.csv", "-b", "key.csv", "-o", "counts%d.csv" % world]
                if world == 1:
                    cmd = [sys.executable, "-m", "tagdigger_b200.tagdigger_script"] + argv
                else:
                    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                           "--master-addr", "127.0.0.1", "--master-port", "29534",
                           "--log-dir", os.path.join(tmp, "logs"), "--redirects", "1",     # every rank's stdout to a file
                           "-m", "tagdigger_b200.tagdigger_script"] + argv
                p = subprocess.run(cmd, cwd=tmp, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, universal_newlines=True)
                path = os.path.join(tmp, "counts%d.csv" % world)
                outs[world] = open(path, "rb").read() if p.returncode == 0 and os.path.exists(path) else None
                stdout[world] = p.stdout if world == 1 else rank0_stdout(os.path.join(tmp, "logs"))
            want = c_oracle.Counter(bcs, tags, "TGCAG").count(fq)[0]
            rows = [ln.split(",")[1:] for ln in outs[1].decode().split("\r\n")[1:] if ln] if outs[1] else []
            ok = (outs[1] is not None and outs[1] == outs[n] and stdout[1] == stdout[n]
                  and np.array(rows, dtype=np.int64).tolist() == want.tolist())
            print("world=%d single file (%s line ends) sharded by byte range: %s" % (n, "CRLF" if newline == b"\r\n" else "LF",
                                                                              "OK" if ok else "MISMATCH"))
            if not ok:
                bad += 1
                print(p.stdout[-2000:] + p.stderr[-2000:])
    return bad


def rank0_stdout(log_dir):
    """Rank 0's stdout under torchrun's ``--log-dir`` (<run>/attempt_0/0/stdout.log)."""
    for root, _dirs, names in os.walk(log_dir):
        if os.path.basename(root) == "0" and "stdout.log" in names:
            with open(os.path.join(root, "stdout.log")) as fh:
                return fh.read()
    return None


if __name__ == "__main__":
    sys.exit(main())
