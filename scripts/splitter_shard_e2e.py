#!/usr/bin/env python3
"""One config-5 library file through the barcode splitter (splitter.split_files) at world 1 and split by W
ranks at once (splitter._split_sharded): every output file of every run must have the md5 of the first
world-1 run's.

The input is the library of scripts/splitter_bgzf_e2e.py (config-5 shape: 150 bp reads in /dev/shm,
96-plex, PstI-MspI-Hall adapters).  W is the number of GPUs present, at least 2: with one GPU the ranks
share it, which checks the protocol but says nothing about whole-box speed.  Each rank runs in its own
process (torch.multiprocessing, gloo for the gathers) on GPU rank % GPUs.  World-1 and world-W runs
alternate, ``runs`` of each (rank 0 alone splits in a world-1 run).  Reported per run: the wall time on
rank 0 between two barriers and, per rank, the seconds of the load (with the line count and the first
gather), pass 1 (sizes), the later gathers and pass 2 (writes); with the GPU's name and power limit and the
host's core count, read in the same run.

    python scripts/splitter_shard_e2e.py [reads] [runs] [out.json]
"""
import contextlib
import hashlib
import io
import json
import os
import pickle
import random
import shutil
import socket
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))

from config5_flow import gpu_name_and_power_limit, make_reads  # noqa: E402
from split_count_shard_e2e import timed  # noqa: E402


def md5s(paths):
    out = []
    for p in paths:
        h = hashlib.md5()
        with open(p, "rb") as fh:
            for chunk in iter(lambda: fh.read(64 << 20), b""):
                h.update(chunk)
        out.append(h.hexdigest())
    return out


def rank_main(rank, world, port, ngpu, key, runs, out_dir):
    import torch.distributed as dist
    from tagdigger_b200 import counting, hostio, splitter
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    device = rank % ngpu
    counting.get_engine(device)
    times = {}
    counting._place_share = timed(times, "load_s", counting._place_share)
    counting._gather_checked = timed(times, "gathers_s", counting._gather_checked)
    splitter._size_share = timed(times, "pass1_s", splitter._size_share)
    splitter._write_share = timed(times, "pass2_s", splitter._write_share)
    adapter = hostio.adapters["PstI-MspI-Hall"]
    outputs = [o for _f, (_b, outs) in key.items() for o in outs]
    with contextlib.redirect_stdout(io.StringIO()):                 # warm-up: module load, buffers
        splitter.split_files({f: [b, outs] for f, (b, outs) in key.items()}, "TGCAG", adapter, maxreads=300000,
                             device=device, rank=rank, world=world, gather=counting.dist_gather)
    results = []
    for run in range(2 * runs):
        w = 1 if run % 2 == 0 else world
        times.clear()
        dist.barrier()
        t0 = time.perf_counter()
        if rank < w:
            with contextlib.redirect_stdout(io.StringIO()):
                splitter.split_files(key, "TGCAG", adapter, device=device, rank=rank, world=w,
                                     gather=counting.dist_gather if w > 1 else None)
        t_done = time.perf_counter()
        dist.barrier()
        t1 = time.perf_counter()
        res = {"run": run, "world": w, "rank": rank, "device": device, "own_s": round(t_done - t0, 4),
               **{k: round(v, 4) for k, v in times.items()}}
        if rank == 0:
            res["wall_s"] = round(t1 - t0, 4)
            res["md5"] = md5s(outputs)
        results.append(res)
        dist.barrier()                                              # rank 0 has read the files
    with open(os.path.join(out_dir, "rank%d.pkl" % rank), "wb") as fh:
        pickle.dump(results, fh)
    dist.barrier()
    dist.destroy_process_group()


def main():
    import numpy as np
    import torch
    import torch.multiprocessing as mp
    from tagdigger_b200 import hostio, synth
    reads = int(sys.argv[1]) if len(sys.argv) > 1 else 8_000_000
    runs = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    out_json = sys.argv[3] if len(sys.argv) > 3 else os.path.join(REPO, "profiles", "r05_splitter_shard_e2e.json")
    ngpu = torch.cuda.device_count()
    if ngpu < 1:
        raise SystemExit("needs a GPU")
    world = max(2, ngpu)
    card = gpu_name_and_power_limit()
    rng = random.Random(5)
    nrng = np.random.default_rng(5)
    barcodes = synth.make_barcodes(96, nrng)
    _, _, seqs = synth.make_marker_pairs(2000, nrng)
    tags = [s for p in seqs for s in p]
    unit = min(reads, 250_000)
    text = make_reads(rng, barcodes, tags, hostio.adapters["PstI-MspI-Hall"], unit)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    tmp = tempfile.mkdtemp(prefix="tdg_split_shard_", dir=os.environ.get("TDG_TMP", base))
    try:
        inp = os.path.join(tmp, "reads.fastq")
        with open(inp, "w") as fh:
            for _ in range(max(1, reads // unit)):
                fh.write(text)
        reads = max(1, reads // unit) * unit
        key = {inp: [barcodes, [os.path.join(tmp, "s%02d.fq" % i) for i in range(len(barcodes))]]}
        ctx = mp.get_context("spawn")
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        procs = [ctx.Process(target=rank_main, args=(r, world, port, ngpu, key, runs, tmp)) for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join()
        if any(p.exitcode != 0 for p in procs):
            raise SystemExit("a rank failed: exit codes %s" % [p.exitcode for p in procs])
        per_rank = []
        for r in range(world):
            with open(os.path.join(tmp, "rank%d.pkl" % r), "rb") as fh:
                per_rank.append(pickle.load(fh))
        input_mb = round(os.path.getsize(inp) / 1e6, 1)
        output_mb = round(sum(os.path.getsize(o) for o in key[inp][1]) / 1e6, 1)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    want = per_rank[0][0]["md5"]
    runs_out = []
    for i, r0 in enumerate(per_rank[0]):
        runs_out.append({"world": r0["world"], "wall_s": r0["wall_s"],
                         "reads_per_s": round(reads / r0["wall_s"], 1), "md5_equal_first_world1_run": r0["md5"] == want,
                         "ranks": [{k: v for k, v in pr[i].items() if k not in ("md5", "wall_s", "run", "world")}
                                   for pr in per_rank[:r0["world"]]]})
    w1 = [r["wall_s"] for r in runs_out if r["world"] == 1]
    ww = [r["wall_s"] for r in runs_out if r["world"] == world]
    res = {"config": "config-5 shape: %d reads (150 bp), PstI-MspI-Hall adapters, 96-plex, one input file" % reads,
           "reads": reads, "input_MB": input_mb, "output_MB": output_mb, "world": world, "gpus": ngpu,
           "ranks_share_one_gpu": world > ngpu, "gpu_and_power_limit": card, "host_cpus": os.cpu_count(),
           "all_md5_equal": all(r["md5_equal_first_world1_run"] for r in runs_out),
           "median_wall_s_world1": sorted(w1)[len(w1) // 2], "median_wall_s_worldW": sorted(ww)[len(ww) // 2],
           "runs": runs_out}
    if world > ngpu:
        res["note"] = "the ranks shared one GPU and one host: a correctness run, the whole-box speed-up is not measured"
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    with open(out_json, "w") as fh:
        json.dump(res, fh, indent=1)
    return 0 if res["all_md5_equal"] else 1


if __name__ == "__main__":
    sys.exit(main())
