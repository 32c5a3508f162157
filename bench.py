#!/usr/bin/env python3
"""Benchmark of the TagDigger counting path on B200 (driver contract).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # the CPU path (oracle port), rank 0 only

Workload = BASELINE.json configs[1]: a 200 M-read single-end GBS FASTQ (100 bp
reads, 96 variable-length barcodes, PstI, 20,000 biallelic marker pairs =
40,000 tags), synthetic, generated directly in HBM by csrc/tdg_synth.cu.  A
"step" is one pass of the counting path over the whole job: zero the count
matrix, count every read, (N > 1) sum the per-GPU matrices with one NCCL
all-reduce.  With N GPUs the reads are sharded N ways (strong scaling).

`value` times the pass with the FASTQ image already resident in HBM; `e2e`
times the same job through tdg_submit from PINNED HOST memory (H2D inside the
timed region) plus the device-to-host read of the count matrix.

`--dump-outputs DIR` writes the count matrix of the last timed step to
DIR/counts.npy (float64, exact for int32 counts; 96 x 40,000 cells = 31 MB).
The reads come from a seeded generator, so two builds given the same arguments
count the same job and their files can be compared cell for cell.
"""

import argparse
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

METRIC = "reads/sec (whole box), 200M-read 96-plex GBS FASTQ"
TOTAL_READS = 200_000_000
NBAR, NPAIRS, READLEN, CUTSITE, SEED = 96, 20000, 100, "TGCAG", 20162


def workload_tables():
    """Barcodes and tags of configs[1] (deterministic)."""
    from tagdigger_b200 import synth
    rng = np.random.default_rng(SEED)
    bcs = synth.make_barcodes(NBAR, rng, cutsite=CUTSITE)
    _, _, seqs = synth.make_marker_pairs(NPAIRS, rng, cutsite=CUTSITE)
    tags = [s for p in seqs for s in p]
    return bcs, tags


def workload_name(nreads):
    return ("configs[1]: %d-read single-end FASTQ (uncompressed image), 96-plex barcodes, "
            "20k biallelic marker pairs (%d tags), PstI, %d bp reads" % (nreads, 2 * NPAIRS, READLEN))


class ClockSampler(object):
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, universal_newlines=True)
        except OSError:
            self.proc = None
        if self.proc is not None:
            time.sleep(0.3)            # nvidia-smi needs a moment before its first sample

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # samples under load = upper half by power
        order = np.argsort(power)
        load = [sm[i] for i in order[len(order) // 2:]]
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


def _oracle_worker(args):
    """One process of the CPU arm: Python restatement of the reference loop."""
    data, bcs, tags = args
    import io
    from oracle import tagdigger_oracle as orc
    prep = orc.prepare(bcs, tags, CUTSITE)
    con = io.TextIOWrapper(io.BytesIO(data), encoding="utf-8", newline=None)
    t0 = time.perf_counter()
    tot = [0, 0, 0]
    orc.count_lines(con, *prep, totals=tot)
    return time.perf_counter() - t0, tot


def cpu_port_rate(sample, nrec, bcs, tags, procs):
    """reads/s of the oracle port on `procs` host processes, each counting its
    own record-aligned shard of the sample (loop time only; the per-process
    trie build is reported separately)."""
    import multiprocessing as mp
    lines = sample.split(b"\n")[:-1]
    per = (nrec + procs - 1) // procs
    shards = []
    for i in range(procs):
        part = lines[4 * per * i: 4 * per * (i + 1)]
        if part:
            shards.append((b"\n".join(part) + b"\n", bcs, tags))
    t0 = time.perf_counter()
    if len(shards) == 1:
        res = [_oracle_worker(shards[0])]
    else:
        with mp.get_context("fork").Pool(len(shards)) as pool:
            res = pool.map(_oracle_worker, shards)
    wall = time.perf_counter() - t0
    loop = max(r[0] for r in res)
    reads = sum(r[1][0] for r in res)
    return reads / loop, len(shards), wall - loop, reads


def verify_slice(eng, gen, bcs, tags, plan, local, nreads, torch):
    """The first `nreads` reads of the job, counted by the CUDA path (tdg_count_device) and by the
    C oracle on the host cores: the matrices and the three totals must be EQUAL."""
    from tagdigger_b200 import _native
    dev, nbytes = gen.generate(local, 0, nreads)
    m2 = torch.zeros((plan.barnum, plan.ntags), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    eng.bind_matrix(m2.data_ptr(), plan.barnum, plan.ntags)
    eng.reset_file()
    eng.count_device(dev, nbytes, 0, _native.TDG_PREV_NONE)
    tot = eng.file_totals()
    got = m2.cpu().numpy().astype(np.int64)
    img = np.empty(nbytes, dtype=np.uint8)
    eng.memcpy_d2h(img.ctypes.data, dev, nbytes)
    gen.free(local, dev)
    t0 = time.perf_counter()
    procs = os.cpu_count() or 1
    from oracle import c_oracle
    want, wtot = c_oracle.count_sharded(img, c_oracle.Counter(bcs, tags, CUTSITE), procs)
    dt = time.perf_counter() - t0
    same = bool((got == want).all()) and [int(x) for x in tot[:3]] == [int(x) for x in wtot]
    return {"ok": same, "reads": int(nreads), "bytes": int(nbytes), "tag_hits": int(want.sum()),
            "oracle": "oracle/oracle.c on %d host processes, %.1f s" % (procs, dt),
            "compared": "count matrix (==, every cell) and [reads, barcode+cutsite, tag] totals"}


def cpu_baseline_leg(args, bcs, tags):
    """cpu_baseline of the N=1 line: the unmodified reference (oracle/_ref) on ONE core over a bounded
    sample; falls back to the Python port when oracle/_ref is not staged."""
    import shutil
    import tempfile
    if _load_reference() is not None:
        tmpdir = tempfile.mkdtemp(prefix="tdg_ref_")
        try:
            rate, build_s, nrec, _ = reference_rate(bcs, tags, 1, args.cpu_sample, 1, 0, tmpdir)
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)
        return {"value": round(rate, 1), "unit": "reads/s", "cores": 1, "kind": "reference",
                "sample": "%d reads of the same workload in one FASTQ file, the UNMODIFIED tagdigger_fun."
                          "find_tags_fastq (oracle/_ref) on one core; its trie build (%.1f s per file, done by the "
                          "reference's own builder) is not in the rate" % (nrec, build_s),
                "trie_build_s": round(build_s, 1), "host_cpus": os.cpu_count()}
    data, _ = host_sample(args.cpu_sample, bcs, tags, SEED + 1)
    rate, procs, build_s, reads = cpu_port_rate(data, args.cpu_sample, bcs, tags, 1)
    return {"value": round(rate, 1), "unit": "reads/s", "cores": 1, "kind": "port",
            "sample": "oracle/_ref not staged: %d reads, Python restatement of find_tags_fastq "
                      "(oracle/tagdigger_oracle.py), loop only; trie build %.1f s extra" % (reads, build_s),
            "host_cpus": os.cpu_count()}


# ---- file -> matrix: the path tagdigger_script users run (tdg_count_file) ---------------------------

def _deflate_piece(job):
    """One piece of a pigz-style single-member gzip stream: raw deflate, ended by a sync flush (or
    finished, for the last piece); returns (compressed bytes, crc32, length)."""
    import zlib
    path, a, b, last, level = job
    with open(path, "rb") as fh:
        fh.seek(a)
        data = fh.read(b - a)
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    out = co.compress(data) + co.flush(zlib.Z_FINISH if last else zlib.Z_SYNC_FLUSH)
    return out, zlib.crc32(data) & 0xFFFFFFFF, len(data)


def _crc32_combine(crc1, crc2, len2):
    """zlib's crc32_combine (not exposed by Python's zlib module)."""
    def times(mat, vec):
        s, i = 0, 0
        while vec:
            if vec & 1:
                s ^= mat[i]
            vec >>= 1
            i += 1
        return s

    def square(mat):
        return [times(mat, mat[n]) for n in range(32)]
    if len2 == 0:
        return crc1
    odd = [0xEDB88320] + [1 << n for n in range(31)]
    even = square(odd)
    odd = square(even)
    while True:
        even = square(odd)
        if len2 & 1:
            crc1 = times(even, crc1)
        len2 >>= 1
        if not len2:
            break
        odd = square(even)
        if len2 & 1:
            crc1 = times(odd, crc1)
        len2 >>= 1
        if not len2:
            break
    return crc1 ^ crc2


def write_gzip_parallel(src, dst, level=6, piece=32 << 20):
    """`src` as ONE gzip member (what gzip/pigz write: a single deflate stream, no index), compressed
    by all host cores in pieces joined with sync flushes."""
    import multiprocessing as mp
    import struct
    size = os.path.getsize(src)
    cuts = list(range(0, size, piece)) + [size]
    jobs = [(src, a, b, b == size, level) for a, b in zip(cuts[:-1], cuts[1:])]
    crc, total = 0, 0
    with mp.get_context("fork").Pool(min(len(jobs), os.cpu_count() or 1)) as pool, open(dst, "wb") as out:
        out.write(b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\x03")
        for blob, c, n in pool.imap(_deflate_piece, jobs):
            out.write(blob)
            crc = _crc32_combine(crc, c, n) if total else c
            total += n
        out.write(struct.pack("<II", crc, total & 0xFFFFFFFF))


def file_legs(args, eng, gen, bcs, tags, plan, local):
    """File -> count matrix on the host through tdg_count_file (the call find_tags_fastq makes): a plain
    FASTQ file (parallel pread into pinned buffers, H2D and counting overlapped) and a single-member
    gzip file of the workload's shape, read from the page cache -- inflated on the device (the
    library's default: the compressed bytes cross PCIe) and, for comparison, by the host threads."""
    import shutil
    import tempfile
    from oracle import c_oracle
    from tagdigger_b200 import _native
    nreads = args.file_reads
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > (16 << 30) else None
    tmpdir = tempfile.mkdtemp(prefix="tdg_bench_", dir=base)
    out = {"reads": nreads, "io_threads": min(int(os.environ.get("TDG_IO_THREADS", "16")), os.cpu_count() or 1),
           "where": "files written just before the run (page cache / %s)" % (base or "tmp")}
    try:
        dev, nbytes = gen.generate(local, 0, nreads)
        img = np.empty(nbytes, dtype=np.uint8)
        eng.memcpy_d2h(img.ctypes.data, dev, nbytes)
        gen.free(local, dev)
        plain = os.path.join(tmpdir, "c2.fq")
        img.tofile(plain)
        want, wtot = c_oracle.count_sharded(img, c_oracle.Counter(bcs, tags, CUTSITE))
        del img
        gz = os.path.join(tmpdir, "c2.fq.gz")
        t0 = time.perf_counter()
        write_gzip_parallel(plain, gz)
        out["gzip_bytes"] = os.path.getsize(gz)
        out["gzip_made_in_s"] = round(time.perf_counter() - t0, 1)
        eng.set_matrix(plan.barnum, plan.ntags)
        for name, path, isgz in (("plain", plain, False), ("gzip", gz, True), ("gzip_host_feed", gz, True)):
            # "gzip": the library's default -- the deflate stream is inflated on the DEVICE (csrc/tdg_gzdev.cuh);
            # "gzip_host_feed": the same file with TDG_GZDEV=0, inflated by the host threads (csrc/tdg_pgz.h)
            if name == "gzip_host_feed":
                os.environ["TDG_GZDEV"] = "0"
            else:
                os.environ.pop("TDG_GZDEV", None)
            best = None
            for rep in range(3 if name != "gzip_host_feed" else 2):
                eng.zero_matrix()
                eng.reset_file()
                t0 = time.perf_counter()
                tot = eng.count_file(path, isgz)
                got = eng.read_matrix()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            same = bool((got == want).all()) and tot[:3] == wtot
            out[name] = {"reads_per_s": round(nreads / best, 1), "text_GBps": round(nbytes / best / 1e9, 2),
                         "seconds": round(best, 3), "exact_vs_c_oracle": "ok" if same else "FAILED"}
        os.environ.pop("TDG_GZDEV", None)
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    return out


def bind_to_gpu_numa(local):
    """Run this rank on the CPUs of the NUMA node its GPU hangs off (sysfs), so that the pinned
    buffers of the end-to-end leg are allocated in memory local to the GPU's PCIe root: with 4-8
    ranks on a two-socket box, buffers on the wrong socket make the H2D copies cross the socket
    link.  Returns a short description for the JSON line."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (getattr(p, "pci_domain_id", 0), p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as fh:
            node = int(fh.read().strip())
        if node < 0:
            return {"gpu_pci": bus, "numa_node": node, "bound": False}
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return {"gpu_pci": bus, "numa_node": node, "bound": False}
        os.sched_setaffinity(0, allowed)
        return {"gpu_pci": bus, "numa_node": node, "bound": True, "cpus": len(allowed)}
    except (OSError, ValueError, AttributeError, RuntimeError) as e:
        return {"bound": False, "why": str(e)[:80]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=TOTAL_READS, help="reads in the whole job")
    ap.add_argument("--e2e-reads", type=int, default=None, help="reads per GPU in the end-to-end leg (default: same job)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=250_000, help="reads the 1-core reference counts for cpu_baseline")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-files", action="store_true")
    ap.add_argument("--file-reads", type=int, default=8_000_000, help="reads in the files of the file -> matrix legs")
    ap.add_argument("--verify-reads", type=int, default=20_000_000,
                    help="reads of the job compared exactly with the C oracle (outside the timed region)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the count matrix of the last timed step to DIR/counts.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours (the reference arm keeps no count matrix)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, world)

    import torch
    import torch.distributed as dist
    from tagdigger_b200 import _native, _synth_native, counting, matchset

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU counting path)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    bcs, tags = workload_tables()
    plan = matchset.plan(bcs, tags, CUTSITE)
    eng = _native.Engine(device=local)
    matrix = torch.zeros((plan.barnum, plan.ntags), dtype=torch.int32, device="cuda")
    eng.set_tags(plan.tags.patterns, plan.tags.index, any_base=plan.tags.any_base)
    eng.bind_matrix(matrix.data_ptr(), plan.barnum, plan.ntags)
    eng.begin_file(plan.bar.patterns, plan.bar.index, plan.bar_tag_off, any_base=plan.bar.any_base)
    if world > 1:
        # the library's own communicator: the all-reduce runs on the counting stream (tdg_allreduce_matrix);
        # torch.distributed only carries the 128-byte id to the ranks
        ids = [eng.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        eng.comm_init(ids[0], world, rank)

    per = args.reads // world
    first = rank * per
    nreads = per if rank < world - 1 else args.reads - first
    gen = _synth_native.Generator(bcs, tags, CUTSITE, readlen=READLEN, seed=SEED)
    expected = torch.zeros_like(matrix)
    dev, nbytes = gen.generate(local, first, nreads, expected.data_ptr())
    torch.cuda.synchronize()

    tstream = torch.cuda.current_stream().cuda_stream

    def step():
        eng.zero_matrix()
        eng.count_device(dev, nbytes, 0, _native.TDG_PREV_NONE)
        if world > 1:
            eng.allreduce_matrix()                  # one ncclAllReduce in stream order behind the last count kernel

    # clocks are sampled over the warm-up and the timed steps (identical work; a timed region of
    # tens of milliseconds alone would give nvidia-smi time for one or two samples)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        step()
    eng.sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()

    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.timing_begin()
    ev0.record()
    eng.stream_wait(tstream)
    for _ in range(args.steps):
        step()
    eng.other_stream_wait(tstream)
    ev1.record()
    torch.cuda.synchronize()
    kernel_ms, ktimed = eng.timing_end()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = args.reads / (ms_per_step * 1e-3)

    # ---- sanity: the counts of the last step ------------------------------------
    tot = eng.file_totals()          # accumulated over warmup + steps on this rank
    nsteps_total = args.warmup + args.steps
    reads_seen = tot[0] // nsteps_total
    p_bar = tot[1] / max(tot[0], 1)
    p_tag = tot[2] / max(tot[0], 1)
    msum = int(matrix.sum(dtype=torch.int64).item())
    exp_t = expected.clone()
    if world > 1:
        dist.all_reduce(exp_t)
        tt = torch.tensor([tot[2] // nsteps_total], dtype=torch.int64, device="cuda")
        dist.all_reduce(tt)
        tag_hits = int(tt.item())
    else:
        tag_hits = tot[2] // nsteps_total
    ok = bool((matrix >= exp_t).all().item()) and msum == tag_hits and reads_seen == nreads
    check = "ok" if ok else "FAILED"
    if rank == 0 and args.dump_outputs:
        # before the legs below, which count into the same matrix
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "counts.npy"), matrix.cpu().numpy().astype(np.float64))

    # ---- roofline of the count kernel (rank 0's launches) --------------------------
    peaks = {}
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    rec_bytes = nbytes / nreads
    alg_per_read = rec_bytes + 32.0 * p_bar + 8.0 * p_tag          # SURVEY 8(d): R + 32 p + 8 h
    alg_bytes = alg_per_read * nreads
    k_ms = kernel_ms / max(ktimed, 1)
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(REPO, "profiles", "traffic.json")) as fh:
            tj = json.load(fh)
        # measured per launch with ncu on a smaller launch of the same workload
        # (profiles/traffic.json); the kernel streams, so DRAM bytes scale with reads
        traffic = int(round(float(tj["dram_bytes_per_read"]) * nreads))
    except (OSError, ValueError, KeyError):
        pass
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic,
                "kernel": "count_kernel<true> (+verify_kernel, fix pass) per launch group",
                "kernel_ms": round(k_ms, 4), "algorithmic_bytes_per_read": round(alg_per_read, 2),
                "stream_bytes_per_read": round(rec_bytes, 2), "peak_source": peak_src}

    # ---- end to end: pinned host image -> counts on the host --------------------------
    e2e = None
    if not args.no_e2e:
        e2e = e2e_leg(args, eng, gen, dev, nbytes, nreads, first, matrix, world, local, dist, torch, tstream)

    # ---- exact check: a slice of the job against the C oracle (rank 0) -----------------------------
    exact = None
    if rank == 0 and not args.no_verify:
        exact = verify_slice(eng, gen, bcs, tags, plan, local, min(args.verify_reads, nreads), torch)
        if not exact["ok"]:
            ok = False
            check = "FAILED"
        eng.bind_matrix(matrix.data_ptr(), plan.barnum, plan.ntags)

    # ---- file -> matrix through tdg_count_file (N = 1 only) ------------------------------------------
    files = None
    if rank == 0 and world == 1 and not args.no_files:
        files = file_legs(args, eng, gen, bcs, tags, plan, local)
        if any(isinstance(v, dict) and v.get("exact_vs_c_oracle") == "FAILED" for v in files.values()):
            ok = False
            check = "FAILED"
        eng.bind_matrix(matrix.data_ptr(), plan.barnum, plan.ntags)
        eng.begin_file(plan.bar.patterns, plan.bar.index, plan.bar_tag_off, any_base=plan.bar.any_base)

    # ---- CPU baseline (rank 0, N = 1 only): the unmodified reference on one core --------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_leg(args, bcs, tags)

    if rank == 0:
        out = {"metric": METRIC, "value": round(value, 1), "unit": "reads/s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8 text -> 2-bit keys, int32 counts",
               "data": "synthetic",
               "config": {"workload": workload_name(args.reads), "reads_per_gpu": nreads,
                          "bytes_per_gpu": nbytes, "l2": "input per GPU far larger than the 126 MB L2; no flush needed",
                          "sharding": "reads split %d ways, one ncclAllReduce of the %dx%d int32 matrix per step on the counting stream (tdg_allreduce_matrix)"
                                      % (world, plan.barnum, plan.ntags) if world > 1 else "single GPU"},
               "gpu_launches": launches, "check": check, "check_exact": exact, "clocks": clocks, "roofline": roofline,
               "e2e": e2e, "e2e_files": files, "cpu_baseline": cpu, "numa": numa}
        print(json.dumps(out))
    gen.free(local, dev)
    if world > 1:
        dist.destroy_process_group()
    return 0 if ok else 1


def e2e_leg(args, eng, gen, dev, nbytes, nreads, first, matrix, world, local, dist, torch, tstream):
    """The same job from pinned host memory: tdg_submit (H2D + kernels,
    pipelined), tdg_end_file, all-reduce, D2H of the matrix -- every step."""
    from tagdigger_b200 import _native
    want = nreads if args.e2e_reads is None else min(args.e2e_reads, nreads)
    if want < nreads:
        gen.free(local, dev)
        dev, nbytes = gen.generate(local, first, want)
    host = None
    size = nbytes
    try:
        host = eng.host_alloc(size)
    except _native.TdgError:
        return {"value": None, "unit": "reads/s", "error": "pinned host allocation of %d bytes failed" % size}
    eng.memcpy_d2h(host, dev, size)
    out = np.empty((eng.rows, eng.cols), dtype=np.int32)
    steps = max(1, min(args.steps, 3))

    def estep():
        eng.zero_matrix()
        eng.reset_file()
        eng.submit((host, size))
        eng.end_file()
        if world > 1:
            eng.allreduce_matrix()
        eng.read_matrix(out)

    estep()                                    # warm-up (allocates the staging slots)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        estep()
    eng.sync()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    nr = torch.tensor([want, size, out.nbytes], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(nr)                      # whole-job totals over all ranks
    dt = float(t.item())
    total_reads, total_h2d, total_d2h = (int(x) for x in nr.tolist())
    eng.host_free(host)
    return {"value": round(total_reads * steps / dt, 1), "unit": "reads/s",
            "h2d_bytes_per_step": total_h2d, "d2h_bytes_per_step": total_d2h,
            "h2d_GBps_per_gpu": round(total_h2d * steps / dt / world / 1e9, 1),
            "steps": steps, "reads_per_step": total_reads, "ms_per_step": round(dt / steps * 1e3, 3),
            "timing": "host wall clock between device synchronisations, max over ranks",
            "path": "tdg_submit from pinned host memory in 64 MiB pieces (H2D overlapped with kernels) + tdg_read_matrix"}


# ---- the reference itself (oracle/_ref, staged by oracle/stage_ref.py) ---------------------------

_REF = {"mod": None, "build_s": 0.0, "memo": {}}


def _load_reference():
    """The UNMODIFIED reference module from oracle/_ref with its trie builder memoised: the
    reference rebuilds both index tries inside every find_tags_fastq call (tagdigger_fun.py:
    218,233: 43 s and 0.9 GB for the 40,000 tags of this workload, paid once per FILE in a real
    run); the harness keeps the tries the reference's own builder returned and hands them back
    on later calls with the same arguments, so that a step times the reference's per-read
    loop.  The build time is reported separately."""
    if _REF["mod"] is not None:
        return _REF["mod"]
    from oracle import stage_ref
    mod = stage_ref.import_ref()
    if mod is None:
        return None
    original = mod.build_sequence_tree

    def build_sequence_tree(sequences, numseq):
        key = (tuple(sequences), numseq)
        tree = _REF["memo"].get(key)
        if tree is None:
            t0 = time.perf_counter()
            tree = original(sequences, numseq)
            _REF["build_s"] += time.perf_counter() - t0
            _REF["memo"][key] = tree
        return tree
    mod.build_sequence_tree = build_sequence_tree
    _REF["mod"] = mod
    return mod


def _reference_worker(job):
    """One host process of the CPU arm: the reference's find_tags_fastq on its own FASTQ shard."""
    import contextlib
    path, bcs, tags = job
    mod = _load_reference()
    with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):
        t0 = time.perf_counter()
        counts = mod.find_tags_fastq(path, bcs, tags, cutsite=CUTSITE)
        dt = time.perf_counter() - t0
    return dt, sum(sum(row) for row in counts)


def host_sample(nreads, bcs, tags, seed):
    """FASTQ text of the workload's shape from the HOST generator (numpy only: the CPU arm maps
    none of the repo's libraries)."""
    from tagdigger_b200 import synth
    rng = np.random.default_rng(seed)
    data, truth = synth.make_fastq(nreads, bcs, tags, rng, cutsite=CUTSITE, readlen=READLEN)
    return data, int(truth["expected"].sum())


def reference_rate(bcs, tags, procs, per_proc, rounds, warm, tmpdir):
    """reads/s of the unmodified reference on `procs` forked host processes, each running
    find_tags_fastq over its own `per_proc`-read file.  Returns (mean rate over `rounds`,
    trie build seconds, reads per round, lower bound check)."""
    import gc
    import multiprocessing as mp
    mod = _load_reference()
    nshard = min(procs, 8)                       # distinct shards; processes beyond that reuse them
    data, _ = host_sample(nshard * per_proc, bcs, tags, SEED + 1)
    lines = data.split(b"\n")[:-1]
    paths = []
    for i in range(nshard):
        path = os.path.join(tmpdir, "shard%d.fq" % i)
        with open(path, "wb") as fh:
            fh.write(b"\n".join(lines[4 * per_proc * i: 4 * per_proc * (i + 1)]) + b"\n")
        paths.append(path)
    empty = os.path.join(tmpdir, "empty.fq")
    open(empty, "wb").close()
    _reference_worker((empty, bcs, tags))          # builds both tries with the reference's builder (timed)
    build_s = _REF["build_s"]
    jobs = [(paths[i % nshard], bcs, tags) for i in range(procs)]
    rates = []
    hits = 0
    if procs == 1:
        for i in range(warm + rounds):
            dt, hits = _reference_worker(jobs[0])
            if i >= warm:
                rates.append(per_proc / dt)
    else:
        gc.freeze()                                # forked children share the tries copy-on-write
        with mp.get_context("fork").Pool(procs) as pool:
            for i in range(warm + rounds):
                res = pool.map(_reference_worker, jobs, chunksize=1)
                if i >= warm:
                    rates.append(procs * per_proc / max(r[0] for r in res))
                hits = res[0][1]
    return float(np.mean(rates)), build_s, procs * per_proc, hits


def usable_procs(per_proc_gb=2.0):
    """Host processes for the CPU arm: every core, unless memory says otherwise (each process may
    end up with its own copy of the 0.9 GB tag trie)."""
    procs = os.cpu_count() or 1
    try:
        import psutil
        avail = psutil.virtual_memory().available / 2.0 ** 30
        procs = max(1, min(procs, int(avail * 0.6 / per_proc_gb)))
    except ImportError:
        pass
    return procs


def reference_arm(args, world):
    """CPU arm: the unmodified reference (oracle/_ref, staged from $TAGDIGGER_REFERENCE by
    oracle/stage_ref.py) on all host cores, each step a bounded sample of the same workload."""
    import shutil
    import tempfile
    bcs, tags = workload_tables()
    tmpdir = tempfile.mkdtemp(prefix="tdg_ref_")
    try:
        if _load_reference() is not None:
            procs = usable_procs()
            per_proc = 50000
            value, build_s, nrec, hits = reference_rate(bcs, tags, procs, per_proc, args.steps, args.warmup, tmpdir)
            kind = "reference"
            sample = ("%d reads of the same workload per step, one %d-read FASTQ file per process, %d forked "
                      "processes each running the UNMODIFIED tagdigger_fun.find_tags_fastq (oracle/_ref); the "
                      "reference's own trie build (%.1f s per file, tagdigger_fun.py:218,233) is done once and "
                      "reused across steps, all other per-call work is timed; %d tag hits in the first shard"
                      % (nrec, per_proc, procs, build_s, hits))
        else:
            procs = os.cpu_count() or 1
            data, _ = host_sample(procs * 40000, bcs, tags, SEED + 1)
            nrec = procs * 40000
            rates = []
            for i in range(args.warmup + args.steps):
                rate, procs, build_s, _ = cpu_port_rate(data, nrec, bcs, tags, procs)
                if i >= args.warmup:
                    rates.append(rate)
            value = float(np.mean(rates))
            kind = "port"
            sample = ("oracle/_ref is not staged on this box: Python restatement of find_tags_fastq "
                      "(oracle/tagdigger_oracle.py), %d reads per step over %d processes, loop only" % (nrec, procs))
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    ms = nrec / value * 1e3
    out = {"impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": "reads/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "python str", "data": "synthetic",
           "config": {"workload": workload_name(args.reads)},
           "cpu_baseline": {"value": round(value, 1), "unit": "reads/s", "cores": procs, "kind": kind,
                            "sample": sample, "host_cpus": os.cpu_count()},
           "e2e": {"value": round(value, 1), "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
