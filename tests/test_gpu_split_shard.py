"""One library file split by several ranks at once: tdg_split_device against tdg_split_block on the same
bytes (both its modes), an allocation-failure sweep over the two passes, and split_files at world 2 and 3
with torch.multiprocessing ranks sharing device 0 and gloo for the gathers, against the world-1 run in this
process: every output file byte for byte, rank 0's output, and exceptions."""

import contextlib
import gzip
import hashlib
import io
import os
import pickle
import random

import numpy as np
import pytest

from feed_check import bgzf_compress
from split_count_check import make_reads, make_tags
from tagdigger_b200 import _native, counting, hostio, splitter
from test_gpu_split_count_shard import BARCODES, HALL, TIMEOUT, _free_port, _records

pytestmark = pytest.mark.gpu

OUTS = ["A.fq", "B.fq", "C.fq", "D.fq", "E.fq"]


@pytest.fixture(scope="module")
def library():
    rng = random.Random(31)
    tags = make_tags(rng, "TGCAG", 60)
    return rng, make_reads(rng, BARCODES, "TGCAG", tags, HALL, 3000)


def _with_host_blocks(text, start=900, step=401):
    recs = _records(text)
    for i in range(start, len(recs), step):                 # records the host cuts
        c1, s, c2, q = recs[i].split("\n")[:4]
        recs[i] = "\n".join([c1, s[:20] + "é" + s[20:], c2, q]) + "\n"
    return recs


def _set_up(eng, barcodes=BARCODES, cutsite="TGCAG", adapter=HALL):
    with contextlib.redirect_stdout(io.StringIO()):
        splitter._load_split(eng, splitter._split_patterns(barcodes, cutsite), barcodes, cutsite, adapter)


@pytest.mark.parametrize("call_bytes", [1500, 40000, 64 << 20])
def test_device_entry_equals_host_entry(library, call_bytes):
    """split_device (from odd device offsets) and split_block (from host memory) on the same walk: equal
    records, consumed bytes, needs_host, bytes of every barcode and flags per call; the sizes-only call's
    offsets and totals equal the full call's."""
    _rng, text = library
    recs = _with_host_blocks(text)
    data = ("".join(recs) + "@x\nACGTATGCAG").encode("utf-8")
    eng = _native.Engine(0)
    try:
        _set_up(eng)
        dev, _ = eng.upload(b"abc" + data)
        try:
            host = np.frombuffer(data, dtype=np.uint8)
            n, pos, size, calls, hosted = len(data), 0, call_bytes, 0, 0
            while pos < n:
                size = min(size, n - pos)
                final = pos + size == n
                r, u, h, pieces, flags = eng.split_block(host[pos:].ctypes.data, size, final, 1 << 40)
                want = (r, u, h, None if pieces is None else [bytes(p) for p in pieces],
                        None if flags is None else flags.tobytes())
                sr, su, sh, offs, sflags, stot = eng.split_device(dev + 3 + pos, size, final, 1 << 40, sizes_only=True)
                assert (sr, su, sh, sflags) == (r, u, h, None)
                dr, du, dh, dpieces, dflags, dtot = eng.split_device(dev + 3 + pos, size, final, 1 << 40)
                got = (dr, du, dh, None if dpieces is None else [bytes(p) for p in dpieces],
                       None if dflags is None else dflags.tobytes())
                assert got == want, pos
                if r and not h:
                    fl = np.frombuffer(want[4], dtype=np.uint8)
                    sums = [len(fl), int(np.count_nonzero(fl & 1)), int(np.count_nonzero(fl & 2))]
                    assert dtot == sums and stot == sums
                    assert offs[0] == 0 and np.diff(offs.astype(np.int64)).tolist() == [len(p) for p in want[3]]
                else:
                    assert offs is None and dtot == [0, 0, 0] and stot == [0, 0, 0]
                if r == 0:
                    if final:
                        break
                    size *= 2                                 # a record longer than the call
                    continue
                calls += 1
                hosted += h
                pos += u
                size = call_bytes
            assert calls >= 1 and hosted >= 1
            eng.split_bgzf(True)
            with pytest.raises(_native.TdgError) as e:
                eng.split_device(dev + 3, 1500, False, 1 << 40, sizes_only=True)
            assert e.value.code == _native.TDG_ERR_STATE
            with pytest.raises(_native.TdgError) as e:
                eng.split_device(dev + 3, 1500, False, 1 << 40)
            assert e.value.code == _native.TDG_ERR_STATE
        finally:
            eng.device_free(dev)
    finally:
        eng.close()


def _two_passes(eng, data, out_dir):
    """Both passes of a sharded split over ``data`` (3 bytes into its allocation) as one rank of one:
    (sizes, totals, output files, progress lines)."""
    _set_up(eng)
    dev, n = eng.upload(b"abc" + data)
    try:
        args = (eng, dev + 3, n - 3, 1 << 40, "lib.fq", BARCODES, [len(b) for b in BARCODES], 5)
        sizes, tot = splitter._size_share(*args)
        paths = [os.path.join(out_dir, o) for o in OUTS]
        for p in paths:
            open(p, "wb").close()
        lines = []
        ends = splitter._write_share(*args, paths, [0] * len(OUTS), [0, 0, 0], lines.append)
    finally:
        eng.device_free(dev)
    return sizes, tot, ends, [open(p, "rb").read() for p in paths], lines


def test_allocation_failure_sweep(library, monkeypatch, tmp_path):
    """TDG_FAIL_ALLOC=k over the two passes (calls of 60 kB, one of them cut by the host): every failure is
    TDG_ERR_NOMEM, and the passes run again equal the run without a failure."""
    monkeypatch.setattr(splitter, "RESIDENT_CALL_BYTES", 60000)
    monkeypatch.setattr(splitter, "BLOCK_READS", 200)
    _rng, text = library
    data = "".join(_with_host_blocks(text, 700, 10 ** 6)).encode("utf-8")
    monkeypatch.delenv("TDG_FAIL_ALLOC", raising=False)
    eng = _native.Engine(0)
    want = _two_passes(eng, data, str(tmp_path))
    eng.close()
    assert want[1][0] == 3000 and want[0] == want[2]
    for k in range(1, 121):
        monkeypatch.setenv("TDG_FAIL_ALLOC", str(k))
        eng = _native.Engine(0)
        failed = False
        try:
            got = _two_passes(eng, data, str(tmp_path))
        except _native.TdgError as e:
            assert e.code == _native.TDG_ERR_NOMEM and "simulated" in e.message, (k, e.code, e.message)
            failed = True
            got = _two_passes(eng, data, str(tmp_path))
        eng.close()
        assert got == want, k
        if not failed:
            break
    else:
        pytest.fail("every one of 120 runs met a simulated failure")
    assert k > 5, k


# ---- split_files at world 2 and 3 --------------------------------------------------------------

def _cases(root, library):
    """{name: (directory, {input: [barcodes, output names]}, cutsite, adapter name, maxreads, bgzf,
    resident call bytes, failure injected on rank 1)}."""
    rng, text = library
    recs = _records(text)
    cases = {}

    def add(name, files, barcodes=BARCODES, cutsite="TGCAG", adapter="PstI-MspI-Hall", maxreads=500000000, bgzf=False,
            call_bytes=None, inject=None):
        d = os.path.join(root, name.replace(" ", "_").replace("'", ""))
        os.makedirs(d)
        key = {}
        for i, (f, data) in enumerate(sorted(files.items())):
            with open(os.path.join(d, f), "wb") as fh:
                fh.write(data if isinstance(data, bytes) else data.encode("utf-8"))
            key[f] = [barcodes, ["%d_%s%s" % (i, o, ".gz" if bgzf else "") for o in OUTS[:len(barcodes)]]]
        cases[name] = (d, key, cutsite, adapter, maxreads, bgzf, call_bytes, inject)

    add("lf", {"lib.fq": text})
    add("crlf", {"lib.fq": text.replace("\n", "\r\n")}, call_bytes=40000)
    mixed = list(recs)
    for i in range(len(mixed) // 2 + 50, len(mixed), 97):       # non-ASCII sequence and quality lines in rank 1's range
        c1, s, c2, q = mixed[i].split("\n")[:4]
        mixed[i] = "\n".join([c1, s[:20] + "é" + s[20:], c2, "ß" + q if i % 2 else q]) + "\n"
    add("non-ascii", {"lib.fq": "".join(mixed)}, call_bytes=40000)
    add("maxreads inside rank 1", {"lib.fq": text}, maxreads=len(recs) * 3 // 4)
    add("bgzf input", {"lib.fq.gz": bgzf_compress(text.encode("utf-8"), block=20000)})
    add("gzip input", {"lib.fq.gz": gzip.compress(text.encode("utf-8"))})
    tags = make_tags(rng, "TGCAG", 20)
    add("more files than ranks", {"%s.fq" % c: make_reads(rng, BARCODES, "TGCAG", tags, HALL, 300) for c in "abcd"})
    add("bgzf output", {"lib.fq": text}, bgzf=True)
    add("lone cr", {"lib.fq": text.replace("\n", "\r")})
    add("load fails on rank 1", {"lib.fq": text}, inject="load")
    for name in sorted(hostio.adapters):
        site = hostio.enzymes[name[:name.find("-")]]
        r2 = random.Random(len(name) * 17)
        t2 = make_tags(r2, site, 50)
        add("adapter " + name, {"lib.fq": make_reads(r2, BARCODES[:4], site, t2, hostio.adapters[name], 3000)},
            barcodes=BARCODES[:4], cutsite=site, adapter=name)
    bad = "".join(mixed).encode("utf-8")
    at = bad.index("é".encode("utf-8"), len(bad) * 11 // 20)       # in rank 1's range at world 2 and 3
    add("invalid utf-8", {"lib.fq": bad[:at] + b"\xff" + bad[at + 2:]})
    return cases


def _outputs(key, out_dir):
    return {f: [b, [os.path.join(out_dir, o) for o in outs]] for f, (b, outs) in key.items()}


def _md5s(d, key, out_dir):
    """md5 of every output file split_files wrote under ``out_dir``."""
    md5 = {}
    for _f, (_b, outs) in _outputs(key, out_dir).items():
        for o in outs:
            p = os.path.join(d, o)
            if os.path.exists(p):
                md5[os.path.basename(o)] = hashlib.md5(open(p, "rb").read()).hexdigest()
    return md5


def _run(d, key, cutsite, adapter, maxreads, bgzf, out_dir, **kw):
    """split_files in directory ``d`` writing under ``out_dir``: (output, exception)."""
    old = os.getcwd()
    os.chdir(d)
    os.makedirs(out_dir, exist_ok=True)
    key = _outputs(key, out_dir)
    out = io.StringIO()
    err = None
    try:
        with contextlib.redirect_stdout(out):
            splitter.split_files(key, hostio.enzymes[adapter[:adapter.find("-")]] if cutsite is None else cutsite,
                                 hostio.adapters[adapter], maxreads=maxreads, bgzf=bgzf, device=0, **kw)
    except Exception as e:  # noqa: BLE001
        err = (type(e).__name__, str(e))
    finally:
        os.chdir(old)
    return out.getvalue(), err


def _rank_main(rank, world, port, cases, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    counting.SHARD_MIN_BYTES = 1024

    def fail(*args, **kw):
        raise _native.TdgError(_native.TDG_ERR_NOMEM, "injected failure")

    results = {}
    for name, (d, key, cutsite, adapter, maxreads, bgzf, call_bytes, inject) in sorted(cases.items()):
        splitter.RESIDENT_CALL_BYTES = call_bytes or (1 << 30)
        with pytest.MonkeyPatch.context() as mp:
            if rank == 1 and inject == "load":
                mp.setattr(counting, "_load_range", fail)
            results[name] = _run(d, key, cutsite, adapter, maxreads, bgzf, "w%d" % world, rank=rank, world=world,
                                 gather=counting.dist_gather)
    with open(os.path.join(out_dir, "rank%d.pkl" % rank), "wb") as fh:
        pickle.dump(results, fh)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_split_equals_one_rank(world, tmp_path, library):
    import torch.multiprocessing as mp
    cases = _cases(str(tmp_path), library)
    want = {name: _run(d, key, cutsite, adapter, maxreads, bgzf, "w1")
            for name, (d, key, cutsite, adapter, maxreads, bgzf, _cb, _inject) in cases.items()}
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, cases, str(tmp_path))) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(TIMEOUT)
    hung = [r for r, p in enumerate(procs) if p.is_alive()]
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert not hung, "ranks %s did not finish" % hung
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    got = []
    for r in range(world):
        with open(str(tmp_path / ("rank%d.pkl" % r)), "rb") as fh:
            got.append(pickle.load(fh))
    dealt = ("gzip input", "more files than ranks", "bgzf output")
    for name, (out, err) in sorted(want.items()):
        d, key = cases[name][:2]
        kinds = [g[name][1] for g in got]
        if name == "invalid utf-8":
            assert err is not None and err[0] == "UnicodeDecodeError", err
            assert kinds[1] is not None and kinds[1][0] == "UnicodeDecodeError", kinds
            assert all(k[0] == "RuntimeError" and "rank 1 " in k[1] for i, k in enumerate(kinds) if i != 1), kinds
            continue
        assert err is None, (name, err)
        assert all(k is None for k in kinds), (name, kinds)
        md5 = _md5s(d, key, "w1")
        assert len(md5) == sum(len(outs) for _b, outs in key.values()), name
        assert _md5s(d, key, "w%d" % world) == md5, name
        if name in dealt:                              # dealt whole: each file's lines on the rank that split it
            assert sorted(sum((g[name][0].splitlines() for g in got), [])) == sorted(out.splitlines()), name
        else:
            assert got[0][name][0] == out, name
            assert all(g[name][0] == "" for g in got[1:]), name
