#!/usr/bin/env python3
"""One config-5 library file counted in one pass (count_files(..., adapter=...)) at world 1 and sharded
across W ranks (counting._count_sharded): every cell of the W-rank matrix must equal the world-1 matrix.

The input is the config-5 shape of scripts/config5_flow.py (150 bp reads in /dev/shm, 96-plex,
PstI-MspI-Hall, 2,000 of 4,000 tags kept).  W is the number of GPUs present, at least 2: with one GPU
the ranks share it, which checks the protocol but says nothing about whole-box speed.  Each rank runs in
its own process (torch.multiprocessing, gloo for the gathers); the matrix sum is the library's NCCL
all-reduce when every rank has a GPU of its own, a CPU all-reduce over gloo otherwise.  Reported per
rank: the seconds of the range load, the line count, the gathers, the one-pass count of the owned
text and the reduce; with the GPU's name and power limit.

With --bgzf the library is bgzipped (members of 65,280 bytes of text, as bgzip writes them) and counted in
both modes: the plain mode with a config-2 tag table (40,000 tags) and the adapter mode as above.  Each is
counted at world 1 (the device gzip feed inflates the file whole) and sharded by member ranges at world W;
reported per rank in addition: the seconds of the member index (tdg_bgzf_index), of the device inflate
(tdg_bgzf_inflate_device), of the plain mode's count (tdg_count_device), and the sum of rank 0's matrix.

    python scripts/split_count_shard_e2e.py [--bgzf] [reads] [out.json]
"""
import contextlib
import io
import json
import os
import pickle
import random
import socket
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))
import numpy as np  # noqa: E402

from config5_flow import gpu_name_and_power_limit, make_reads  # noqa: E402


def timed(times, key, fn):
    def run(*a, **k):
        t0 = time.perf_counter()
        try:
            return fn(*a, **k)
        finally:
            times[key] = times.get(key, 0.0) + time.perf_counter() - t0
    return run


def bgzip(src, dst):
    """``src`` as BGZF (one member per 65,280 bytes, compressed by a pool of processes, then the EOF marker)."""
    import multiprocessing
    from feed_check import bgzf_block
    with open(src, "rb") as fh:
        data = fh.read()
    pieces = [data[i:i + 65280] for i in range(0, len(data), 65280)]
    with multiprocessing.Pool() as pool:
        blocks = pool.starmap(bgzf_block, [(p, 1) for p in pieces], chunksize=256)
    with open(dst, "wb") as fh:
        fh.writelines(blocks)
        fh.write(bgzf_block(b""))


def rank_main(rank, world, port, ngpu, key, tags, out_dir, adapter="PstI-MspI-Hall", tag="x"):
    import torch
    import torch.distributed as dist
    from tagdigger_b200 import _native, counting, splitter
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    device = rank % ngpu
    eng = counting.get_engine(device)
    own_gpu = world <= ngpu
    if own_gpu:
        counting.init_comm(eng, rank, world)

    def cpu_reduce(ptr, rows, cols, e):
        t = torch.from_numpy(e.read_matrix())
        dist.all_reduce(t)
        a = np.ascontiguousarray(t.numpy())
        e.memcpy_h2d(ptr, a.ctypes.data, a.nbytes)

    times = {}
    counting._load_range = timed(times, "load_s", counting._load_range)
    counting._load_bgzf_share = timed(times, "load_s", counting._load_bgzf_share)
    _native.bgzf_index = timed(times, "index_s", _native.bgzf_index)
    _native.Engine.bgzf_inflate_device = timed(times, "inflate_s", _native.Engine.bgzf_inflate_device)
    _native.Engine.count_lines_device = timed(times, "line_count_s", _native.Engine.count_lines_device)
    _native.Engine.count_device = timed(times, "count_s", _native.Engine.count_device)
    splitter.count_trimmed_resident = timed(times, "split_count_s", splitter.count_trimmed_resident)
    gather = timed(times, "gathers_s", counting.dist_gather)
    totals = {}
    reduce = timed(times, "reduce_s", counting.engine_reduce if own_gpu else cpu_reduce)
    dist.barrier()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        _, matrix = counting.count_files(key, tags, "TGCAG", device=device, rank=rank, world=world, reduce=reduce,
                                         gather=gather, as_array=True, adapter=adapter, totals=totals)
    times["count_files_s"] = time.perf_counter() - t0
    res = {"rank": rank, "device": device, **{k: round(v, 4) for k, v in times.items()},
           "holds_file": bool(totals), "matrix_sum": int(matrix.sum())}
    with open(os.path.join(out_dir, "rank%d_%s.pkl" % (rank, tag)), "wb") as fh:
        pickle.dump((res, matrix if rank == 0 else None), fh)
    dist.barrier()
    dist.destroy_process_group()


def main():
    import torch
    import torch.multiprocessing as mp
    from tagdigger_b200 import counting, hostio, synth
    args = [a for a in sys.argv[1:] if a != "--bgzf"]
    use_bgzf = "--bgzf" in sys.argv[1:]
    reads = int(args[0]) if args else 8_000_000
    out_json = args[1] if len(args) > 1 else os.path.join(REPO, "profiles", "r03_split_count_shard_e2e.json")
    ngpu = torch.cuda.device_count()
    if ngpu < 1:
        raise SystemExit("needs a GPU")
    world = max(2, ngpu)
    rng = random.Random(5)
    nrng = np.random.default_rng(5)
    adapter = hostio.adapters["PstI-MspI-Hall"]
    barcodes = synth.make_barcodes(96, nrng)
    names, _, seqs = synth.make_marker_pairs(2000, nrng)
    tags = [s for p in seqs for s in p]
    keep = set(names[::2])
    kept_tags = [s for name, p in zip(names, seqs) if name in keep for s in p]
    unit = 250_000
    text = make_reads(rng, barcodes, tags, adapter, unit)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    tmp = tempfile.mkdtemp(prefix="tdg_shard_", dir=os.environ.get("TDG_TMP", base))
    inp = os.path.join(tmp, "reads.fastq")
    with open(inp, "w") as fh:
        for _ in range(max(1, reads // unit)):
            fh.write(text)
    reads = max(1, reads // unit) * unit
    if use_bgzf:
        sys.path.insert(0, os.path.join(REPO, "tests"))
        return bgzf_legs(inp, tmp, reads, barcodes, tags, kept_tags, ngpu, world, out_json)
    key = {inp: [list(barcodes), ["Sample%02d" % i for i in range(len(barcodes))]]}
    res = {"config": "config 5 shape: %d reads (150 bp), PstI-MspI-Hall adapters, 96-plex, %d tags of which %d kept"
                     % (reads, len(tags), len(kept_tags)),
           "input_MB": round(os.path.getsize(inp) / 1e6, 1), "gpu": gpu_name_and_power_limit(), "gpus": ngpu,
           "world": world, "host_cpus": os.cpu_count()}
    res["ranks_share_one_gpu"] = world > ngpu
    with contextlib.redirect_stdout(io.StringIO()):
        counting.count_files(key, kept_tags, "TGCAG", as_array=True, adapter="PstI-MspI-Hall")      # warm-up
        t0 = time.perf_counter()
        _, want = counting.count_files(key, kept_tags, "TGCAG", as_array=True, adapter="PstI-MspI-Hall")
        res["world1_s"] = round(time.perf_counter() - t0, 3)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(rank_main, args=(world, port, ngpu, key, kept_tags, tmp), nprocs=world, join=True)
    ranks = []
    got = None
    for r in range(world):
        with open(os.path.join(tmp, "rank%d_x.pkl" % r), "rb") as fh:
            info, m = pickle.load(fh)
        ranks.append(info)
        if r == 0:
            got = m
    res["ranks"] = ranks
    res["cells"] = int(want.size)
    res["cells_equal_world1"] = int(np.count_nonzero(got == want))
    res["matrix_equals_world1"] = "ok (every cell)" if np.array_equal(got, want) else "FAILED"
    res["tag_hits"] = int(want.sum())
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    with open(out_json, "w") as fh:
        fh.write(line + "\n")
    for f in os.listdir(tmp):
        os.remove(os.path.join(tmp, f))
    os.rmdir(tmp)
    return 0 if np.array_equal(got, want) else 1


def bgzf_legs(inp, tmp, reads, barcodes, tags, kept_tags, ngpu, world, out_json):
    import torch.multiprocessing as mp
    from tagdigger_b200 import counting, synth
    gz = inp + ".gz"
    t0 = time.perf_counter()
    bgzip(inp, gz)
    bgzip_s = time.perf_counter() - t0
    text_mb = os.path.getsize(inp) / 1e6
    os.remove(inp)
    names, _, seqs = synth.make_marker_pairs(18000, np.random.default_rng(7))
    config2_tags = list(tags) + [s for p in seqs for s in p]            # 4,000 + 36,000 tags
    key = {gz: [list(barcodes), ["Sample%02d" % i for i in range(len(barcodes))]]}
    res = {"config": "%d reads (150 bp, the config-5 generator), 96-plex, bgzipped; plain mode with %d tags (config-2 "
                     "table), adapter mode (PstI-MspI-Hall) with %d kept tags" % (reads, len(config2_tags), len(kept_tags)),
           "text_MB": round(text_mb, 1), "bgzf_MB": round(os.path.getsize(gz) / 1e6, 1), "bgzip_s": round(bgzip_s, 1),
           "gpu": gpu_name_and_power_limit(), "gpus": ngpu, "world": world, "host_cpus": os.cpu_count(),
           "ranks_share_one_gpu": world > ngpu}
    if world > ngpu:
        res["note"] = "ranks share one GPU: a correctness run; whole-box speed-up not measured"
    ok = True
    for leg, adapter, leg_tags in (("plain", None, config2_tags), ("adapter", "PstI-MspI-Hall", kept_tags)):
        out = {}
        with contextlib.redirect_stdout(io.StringIO()):
            counting.count_files(key, leg_tags, "TGCAG", as_array=True, adapter=adapter)          # warm-up
            t0 = time.perf_counter()
            _, want = counting.count_files(key, leg_tags, "TGCAG", as_array=True, adapter=adapter)
            out["world1_s"] = round(time.perf_counter() - t0, 3)
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        t0 = time.perf_counter()
        mp.spawn(rank_main, args=(world, port, ngpu, key, leg_tags, tmp, adapter, leg), nprocs=world, join=True)
        out["worldW_spawn_to_end_s"] = round(time.perf_counter() - t0, 3)
        ranks = []
        for r in range(world):
            with open(os.path.join(tmp, "rank%d_%s.pkl" % (r, leg)), "rb") as fh:
                info, m = pickle.load(fh)
            ranks.append(info)
            if r == 0:
                got = m
        out["ranks"] = ranks
        out["worldW_count_files_s"] = max(r["count_files_s"] for r in ranks)
        out["speedup_count_files"] = round(out["world1_s"] / out["worldW_count_files_s"], 3)
        out["world1_reads_per_s"] = round(reads / out["world1_s"])
        out["cells"] = int(want.size)
        out["matrix_sum_world1"] = int(want.sum())
        out["matrix_equals_world1"] = "ok (every cell)" if np.array_equal(got, want) else "FAILED"
        out["sharded"] = all(r["holds_file"] for r in ranks)
        ok = ok and np.array_equal(got, want)
        res[leg] = out
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    with open(out_json, "w") as fh:
        fh.write(line + "\n")
    for f in os.listdir(tmp):
        os.remove(os.path.join(tmp, f))
    os.rmdir(tmp)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
