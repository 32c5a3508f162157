"""One library file sharded across ranks: tdg_split_count_device against tdg_split_count_block on the
same bytes, and count_files at world 2 and 3, in the plain mode and in the one-pass split-and-count mode
(``adapter=...``), with torch.multiprocessing ranks sharing device 0 and gloo for the gathers and for the
matrix sum, against the world-1 run in this process: samples, matrix, totals, rank 0's output and
exceptions, also when rank 1 fails to load or to count its range."""

import contextlib
import gzip
import io
import os
import pickle
import random
import socket

import numpy as np
import pytest

from split_count_check import make_reads, make_tags
from tagdigger_b200 import _native, counting, hostio, matchset, splitter

pytestmark = pytest.mark.gpu

BARCODES = ["ACGTA", "TTGCAC", "GGAT", "CATCGGA", "AACCGT"]
SAMPLES = ["A", "B", "C", "A", "D"]
HALL = hostio.adapters["PstI-MspI-Hall"]
HEAD_CAP = 8192                 # the children's head cap: a file with longer lines is counted whole
TIMEOUT = 600                   # seconds for all cases of one world


def _records(text):
    lines = text.split("\n")
    return ["\n".join(lines[i:i + 4]) + "\n" for i in range(0, len(lines) - 1, 4)]


@pytest.fixture(scope="module")
def library():
    rng = random.Random(23)
    tags = make_tags(rng, "TGCAG", 60)
    return rng, tags, make_reads(rng, BARCODES, "TGCAG", tags, HALL, 3000)


def _set_up(eng, tags, nrows=4):
    plan = matchset.plan([""], tags, "TGCAG")
    eng.set_tags(plan.tags.patterns, plan.tags.index, any_base=plan.tags.any_base)
    eng.set_matrix(nrows, plan.ntags)
    return plan


@pytest.mark.parametrize("call_bytes", [1500, 40000, 64 << 20])
def test_device_entry_equals_host_entry(library, call_bytes):
    """The same walk over the same bytes, through host memory and through device memory (at offsets
    of any alignment): equal records, consumed bytes, needs_host and totals per call, equal matrix."""
    rng, tags, text = library
    recs = _records(text)
    for i in range(900, len(recs), 401):                    # blocks the host cuts
        c1, s, c2, q = recs[i].split("\n")[:4]
        recs[i] = "\n".join([c1, s[:20] + "é" + s[20:], c2, q]) + "\n"
    data = ("".join(recs) + "@x\nACGTATGCAG").encode("utf-8")
    eng = _native.Engine(0)
    try:
        runs = []
        dev, n = eng.upload(data)
        try:
            for device in (False, True):
                plan = _set_up(eng, tags)
                splitter._trimmed_counter(eng, BARCODES, [0, 1, 2, 0, 3], plan, "TGCAG", HALL)
                host = np.frombuffer(data, dtype=np.uint8)
                calls, pos, size = [], 0, call_bytes
                while pos < n:
                    size = min(size, n - pos)
                    final = pos + size == n
                    if device:
                        r = eng.split_count_device(dev + pos, size, final, 1 << 40)
                    else:
                        r = eng.split_count_block(host[pos:].ctypes.data, size, final, 1 << 40)
                    calls.append(r)
                    if r[0] == 0:
                        if final:
                            break
                        size *= 2                             # a record longer than the call
                        continue
                    pos += r[1]
                    size = call_bytes
                runs.append((calls, eng.read_matrix().tolist()))
        finally:
            eng.device_free(dev)
    finally:
        eng.close()
    assert runs[0] == runs[1]
    calls = runs[0][0]
    assert sum(c[0] for c in calls) == len(recs)
    assert any(c[2] for c in calls)
    hits = sum(c[3][3] for c in calls if c[0] and not c[2])     # a needs_host call leaves the matrix alone
    assert sum(map(sum, runs[0][1])) == hits
    assert hits > 100 or call_bytes >= len(data)


def _resident(eng, data, tags):
    plan = _set_up(eng, tags)
    dev, n = eng.upload(data)
    try:
        tot = splitter.count_trimmed_resident(eng, dev + 3, n - 3, BARCODES, [0, 2, 1, 0, 3], plan, "TGCAG", HALL, 1 << 40)
    finally:
        eng.device_free(dev)
    return eng.read_matrix().tobytes(), tot


def test_allocation_failure_sweep(library, monkeypatch):
    """TDG_FAIL_ALLOC=k over one split_count_device walk (calls of 60 kB, one of them cut by the host):
    every failure is TDG_ERR_NOMEM, and the walk run again equals the run without a failure."""
    monkeypatch.setattr(splitter, "RESIDENT_CALL_BYTES", 60000)
    monkeypatch.setattr(splitter, "BLOCK_READS", 200)
    rng, tags, text = library
    recs = _records(text)
    recs[700] = recs[700].replace("\n", "é\n", 2).replace("é\n", "\n", 1)
    data = ("abc" + "".join(recs)).encode("utf-8")            # the text starts 3 bytes into the allocation
    monkeypatch.delenv("TDG_FAIL_ALLOC", raising=False)
    eng = _native.Engine(0)
    want = _resident(eng, data, tags)
    eng.close()
    assert want[1][0] == len(recs)
    for k in range(1, 121):
        monkeypatch.setenv("TDG_FAIL_ALLOC", str(k))
        eng = _native.Engine(0)
        failed = False
        try:
            got = _resident(eng, data, tags)
        except _native.TdgError as e:
            assert e.code == _native.TDG_ERR_NOMEM and "simulated" in e.message, (k, e.code, e.message)
            failed = True
            got = _resident(eng, data, tags)
        eng.close()
        assert got == want, k
        if not failed:
            break
    else:
        pytest.fail("every one of 120 runs met a simulated failure")
    assert k > 10, k


# ---- count_files at world 2 and 3 --------------------------------------------------------------

def _write(path, text, raw=None):
    data = raw if raw is not None else text.encode("utf-8")
    with open(path, "wb") as fh:
        fh.write(gzip.compress(data) if path.endswith("gz") else data)


def _cases(root, library):
    """{name: (directory, key, tags, cutsite, adapter name, maxreads / split_maxreads, resident call bytes,
    failure injected on rank 1)}."""
    rng, tags, text = library
    recs = _records(text)
    cases = {}

    def add(name, files, key=None, tags_=tags, cutsite="TGCAG", adapter="PstI-MspI-Hall", maxreads=500000000,
            call_bytes=None, inject=None):
        d = os.path.join(root, name.replace(" ", "_"))
        os.makedirs(d)
        for f, t in files.items():
            _write(os.path.join(d, f), t if isinstance(t, str) else None, raw=t if isinstance(t, bytes) else None)
        cases[name] = (d, key or {f: [BARCODES, SAMPLES] for f in files}, tags_, cutsite, adapter, maxreads, call_bytes,
                       inject)

    add("lf", {"lib.fq": text})
    add("lf, calls of 40 kB", {"lib.fq": text}, call_bytes=40000)
    add("load fails on rank 1", {"lib.fq": text}, inject="load")
    add("count fails on rank 1", {"lib.fq": text}, inject="count")
    add("crlf", {"lib.fq": text.replace("\n", "\r\n")}, call_bytes=40000)
    data = text.encode("utf-8")
    shifted = bytearray(data)
    for pos in sorted({data.index(b"\n", len(data) * r // w) + 1 for r, w in ((1, 2), (1, 3), (2, 3))}, reverse=True):
        shifted[pos:pos] = b"\n"                              # a blank line at the nominal cuts of world 2 and 3
    add("blank lines at the cuts", {"lib.fq": shifted.decode("utf-8")})
    add("no final newline", {"lib.fq": text[:-1]})
    add("partial record", {"lib.fq": text + "@x\nACGTATGCAGTT\n"})
    path = os.path.join(root, "first.fq")
    _write(path, text)
    for w in (2, 3):                                           # the limit inside rank 1's range and at its start
        first = _first_record(path, w, 1)
        for m in (first, first + 5):
            add("maxreads %d" % m, {"lib.fq": text}, maxreads=m)
    add("maxreads 7", {"lib.fq": text}, maxreads=7)
    half = len(recs) // 2
    mixed = list(recs)
    for i in range(half + 50, len(mixed), 97):                 # non-ASCII sequence lines in the later ranges
        c1, s, c2, q = mixed[i].split("\n")[:4]
        mixed[i] = "\n".join([c1, s[:20] + "é" + s[20:], c2, "ß" + q if i % 2 else q]) + "\n"
    add("non-ascii", {"lib.fq": "".join(mixed)}, call_bytes=40000)
    other = make_reads(rng, ["CCATG", "ACGTA", "GTTAC"], "TGCAG", tags, HALL, 800)
    add("plain and gzip", {"a.fq": text, "b.fq.gz": other},
        key={"a.fq": [BARCODES, SAMPLES], "b.fq.gz": [["CCATG", "ACGTA", "GTTAC"], ["C", "E", "A"]]})
    add("lone cr", {"lib.fq": text.replace("\n", "\r")})
    giant = "".join("\n".join([c1, s + "ACGT" * 2500, c2, q + "#" * 10000]) + "\n"
                    for c1, s, c2, q in (r.split("\n")[:4] for r in recs[:400]))
    add("giant lines", {"lib.fq": giant})
    for name in sorted(hostio.adapters):
        site = hostio.enzymes[name[:name.find("-")]]
        r2 = random.Random(len(name) * 13)
        t2 = make_tags(r2, site, 50)
        add("adapter " + name, {"lib.fq": make_reads(r2, BARCODES[:4], site, t2, hostio.adapters[name], 3000)},
            key={"lib.fq": [BARCODES[:4], ["S0", "S1", "S2", "S0"]]}, tags_=t2, cutsite=site, adapter=name)
    bad = "".join(mixed).encode("utf-8")
    at = bad.index("é".encode("utf-8"), len(bad) * 11 // 20)       # in rank 1's range at world 2 and 3
    add("invalid utf-8", {"lib.fq": bad[:at] + b"\xff" + bad[at + 2:]})
    return cases


def _first_record(path, world, rank):
    """The index of the first record rank ``rank`` counts when ``path`` is sharded across ``world`` ranks."""
    data = open(path, "rb").read()
    bounds = counting.range_bounds(path, world)
    spans = list(zip(bounds[:-1], bounds[1:]))
    lines = [len(io.StringIO(data[lo:hi].decode("utf-8"), newline=None).readlines()) for lo, hi in spans]
    heads = [counting.range_head(path, lo, hi) for lo, hi in spans]
    return counting.plan_trimmed_shards(lines, heads, 1 << 40)[rank][2]


MODES = ("plain", "adapter")


def _run(mode, key, tags, cutsite, adapter, maxreads, **kw):
    """count_files in the plain mode or with ``adapter``, its output captured: (result, output, exception)."""
    out = io.StringIO()
    tot = {}
    res = err = None
    args = dict(maxreads=maxreads) if mode == "plain" else dict(adapter=adapter, split_maxreads=maxreads)
    try:
        with contextlib.redirect_stdout(out):
            s, m = counting.count_files(key, tags, cutsite, totals=tot, as_array=True, device=0, **args, **kw)
        res = (s, m.tolist(), tot)
    except Exception as e:  # noqa: BLE001
        err = (type(e).__name__, str(e))
    return res, out.getvalue(), err


def _rank_main(rank, world, port, cases, out_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    counting.SHARD_MIN_BYTES = 1024
    counting.HEAD_CAP = HEAD_CAP

    def cpu_reduce(ptr, rows, cols, eng):
        t = torch.from_numpy(eng.read_matrix())
        dist.all_reduce(t)
        a = np.ascontiguousarray(t.numpy())
        eng.memcpy_h2d(ptr, a.ctypes.data, a.nbytes)

    def fail(*args, **kw):
        raise _native.TdgError(_native.TDG_ERR_NOMEM, "injected failure")

    results = {}
    for (name, mode), (d, key, tags, cutsite, adapter, maxreads, call_bytes, inject) in sorted(cases.items()):
        os.chdir(d)
        splitter.RESIDENT_CALL_BYTES = call_bytes or (1 << 30)
        with pytest.MonkeyPatch.context() as mp:
            if rank == 1 and inject == "load":
                mp.setattr(counting, "_load_range", fail)
            if rank == 1 and inject == "count":                 # the own-range count of either mode
                mp.setattr(_native.Engine, "count_device", fail)
                mp.setattr(splitter, "count_trimmed_resident", fail)
            results[name, mode] = _run(mode, key, tags, cutsite, adapter, maxreads, rank=rank, world=world,
                                       reduce=cpu_reduce, gather=counting.dist_gather)
    with open(os.path.join(out_dir, "rank%d.pkl" % rank), "wb") as fh:
        pickle.dump(results, fh)
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_count_equals_one_rank(world, tmp_path, library):
    import torch.multiprocessing as mp
    # the plain mode does not check UTF-8 in a sharded range (DESIGN §7), so that case is the adapter mode's
    cases = {(name, mode): c for name, c in _cases(str(tmp_path), library).items() for mode in MODES
             if mode == "adapter" or name != "invalid utf-8"}
    want = {}
    old = os.getcwd()
    try:
        for (name, mode), (d, key, tags, cutsite, adapter, maxreads, _cb, _inject) in cases.items():
            os.chdir(d)
            want[name, mode] = _run(mode, key, tags, cutsite, adapter, maxreads)
    finally:
        os.chdir(old)
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
    for case, (res, out, err) in sorted(want.items()):
        name, mode = case
        kinds = [g[case][2] for g in got]
        if name == "invalid utf-8":
            assert res is None and err[0] == "UnicodeDecodeError", err
            assert kinds[1][0] == "UnicodeDecodeError", kinds
        if name == "count fails on rank 1":
            assert err is None, err
            assert kinds[1][0] == "TdgError" and "injected" in kinds[1][1], kinds
        if name in ("invalid utf-8", "count fails on rank 1"):      # rank 1 raises its own error, the others name it
            assert all(k[0] == "RuntimeError" and "rank 1 " in k[1] for i, k in enumerate(kinds) if i != 1), kinds
            continue
        assert err is None, (case, err)
        for r in range(world):
            g_res, g_out, g_err = got[r][case]
            assert g_err is None, (case, r, g_err)
            assert g_res[0] == res[0] and g_res[1] == res[1], (case, r)
            for f, t in g_res[2].items():
                assert t == res[2][f], (case, r, f)
        holders = [sorted(got[r][case][0][2]) for r in range(world)]
        # counted whole on rank 0: no cut point, a failed load, and (in the adapter mode, which sends every
        # range's first lines to the other ranks) lines longer than HEAD_CAP
        if name in ("lone cr", "load fails on rank 1") or (name, mode) == ("giant lines", "adapter"):
            assert holders == [["lib.fq"]] + [[]] * (world - 1), case
        elif name != "plain and gzip":                         # sharded: every rank has the file's totals
            assert holders == [["lib.fq"]] * world, case
        if name == "plain and gzip" and world == 2:            # two files, two ranks: dealt whole
            assert sorted(got[0][case][1].splitlines() + got[1][case][1].splitlines()) == sorted(out.splitlines())
        else:
            assert got[0][case][1] == out, case
        if name == "plain and gzip" and world == 3:
            assert all("a.fq" in h for h in holders), holders
