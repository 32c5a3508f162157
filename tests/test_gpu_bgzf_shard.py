"""One BGZF library file sharded across ranks by member ranges: tdg_bgzf_inflate_device against zlib, its
errors and its allocation failures, and count_files at world 2 and 3 (torch.multiprocessing ranks sharing
device 0, gloo for the gathers and the matrix sum) against the world-1 run in this process, in the plain
mode and with ``adapter=...``: samples, matrix, totals, rank 0's output and exceptions, and which ranks
hold the file (every rank when it is sharded, rank 0 alone when it is counted whole)."""

import contextlib
import gzip
import os
import pickle
import random

import numpy as np
import pytest

from feed_check import bgzf_compress
from split_count_check import make_reads, make_tags
from tagdigger_b200 import _native, counting
from test_gpu_split_count_shard import BARCODES, HALL, HEAD_CAP, SAMPLES, TIMEOUT, _free_port, _records, _run

pytestmark = pytest.mark.gpu

BLOCK = 20000                   # bytes of text per member: a few dozen members per library
LOOKAHEAD_CAP = 1 << 20         # the children's look-ahead cap: the 4 MiB line at the cuts passes it at world 2


@pytest.fixture(scope="module")
def library():
    rng = random.Random(29)
    tags = make_tags(rng, "TGCAG", 60)
    return rng, tags, make_reads(rng, BARCODES, "TGCAG", tags, HALL, 3000)


def _bgzf_file(tmp_path, data, name="a.fq.gz"):
    path = str(tmp_path / name)
    with open(path, "wb") as fh:
        fh.write(bgzf_compress(data, block=BLOCK))
    return path


def _inflate(eng, path, c_lo, c_hi, cap):
    dev = eng.device_alloc(max(cap, 1))
    try:
        n, high = eng.bgzf_inflate_device(path, c_lo, c_hi, dev, cap)
        out = np.empty(n, dtype=np.uint8)
        if n:
            eng.memcpy_d2h(out.ctypes.data, dev, n)
    finally:
        eng.device_free(dev)
    return out.tobytes(), high


def test_inflate_device_equals_zlib(tmp_path, library):
    text = library[2].encode("utf-8")
    path = _bgzf_file(tmp_path, text)
    off, isize = _native.bgzf_index(path)
    size = os.path.getsize(path)
    m = len(off)
    assert m > 20 and isize[-1] == 0                          # the end-of-file marker is the last member
    t = np.concatenate([[0], np.cumsum(isize.astype(np.int64))])
    at = [int(x) for x in off] + [size]
    eng = _native.Engine(0)
    try:
        for k0, k1 in [(0, m), (0, 1), (3, 9), (m // 2, m), (m - 2, m), (m - 1, m), (5, 5)]:
            got, high = _inflate(eng, path, at[k0], at[k1], int(t[k1] - t[k0]) + 100)
            assert got == text[t[k0]:t[k1]], (k0, k1)
            assert not high
        uni = _bgzf_file(tmp_path, library[2].replace("ACGTA", "ACGTé", 1).encode("utf-8"), "u.fq.gz")
        got, high = _inflate(eng, uni, 0, os.path.getsize(uni), len(text) + 100)
        assert high and got.decode("utf-8").count("é") == 1
    finally:
        eng.close()


def test_inflate_device_errors(tmp_path, library):
    text = library[2].encode("utf-8")
    path = _bgzf_file(tmp_path, text)
    off, isize = _native.bgzf_index(path)
    size = os.path.getsize(path)
    eng = _native.Engine(0)
    try:
        with pytest.raises(_native.TdgError) as e:                 # cap too small
            _inflate(eng, path, 0, size, len(text) - 1)
        assert e.value.code == _native.TDG_ERR_ARG
        for c_lo, c_hi in [(int(off[2]) + 5, int(off[4])), (int(off[2]), int(off[4]) + 5)]:   # no member start; overrun
            with pytest.raises(_native.TdgError) as e:
                _inflate(eng, path, c_lo, c_hi, len(text))
            assert e.value.code == _native.TDG_ERR_GZIP, (c_lo, c_hi, e.value.message)
        bad = bytearray(open(path, "rb").read())
        bad[int(off[3]) + 40] ^= 0x10                            # a flipped bit in member 3's deflate data
        with open(str(tmp_path / "bad.fq.gz"), "wb") as fh:
            fh.write(bytes(bad))
        with pytest.raises(_native.TdgError) as e:
            _inflate(eng, str(tmp_path / "bad.fq.gz"), 0, size, len(text))
        assert e.value.code == _native.TDG_ERR_GZIP
        got, _ = _inflate(eng, path, 0, size, len(text))          # the context still works
        assert got == text
    finally:
        eng.close()


def test_inflate_device_allocation_failure_sweep(tmp_path, library, monkeypatch):
    """TDG_FAIL_ALLOC=k: every failure is TDG_ERR_NOMEM, and the same context then inflates correctly."""
    text = library[2].encode("utf-8")
    path = _bgzf_file(tmp_path, text)
    size = os.path.getsize(path)
    monkeypatch.setenv("TDG_GZDEV_MAXCHUNKS", "8")              # several rounds
    for k in range(1, 121):
        monkeypatch.setenv("TDG_FAIL_ALLOC", str(k))
        eng = _native.Engine(0)
        failed = False
        try:
            got, _ = _inflate(eng, path, 0, size, len(text))
        except _native.TdgError as e:
            assert e.code == _native.TDG_ERR_NOMEM, (k, e.code, e.message)
            failed = True
            got, _ = _inflate(eng, path, 0, size, len(text))
        eng.close()
        assert got == text, k
        if not failed:
            break
    else:
        pytest.fail("every one of 120 runs met a simulated failure")
    assert k > 5, k


# ---- count_files at world 2 and 3 --------------------------------------------------------------

RAISES = ("invalid utf-8", "corrupt member")     # world 1 raises: rank 0 raises the same, the others reach the reduce


def _cases(root, library):
    """{(name, mode): (directory, key, tags, maxreads, rank-1 inflate fails, environment, expected)} with expected
    'sharded', 'fallback' (rank 0 counts the file whole after the first gather) or 'dealt' (never sharded)."""
    rng, tags, text = library
    recs = _records(text)
    n = len(recs)
    cases = {}

    def add(name, data, expected, modes=("plain", "adapter"), maxreads=500000000, inject=False, env=None, name_gz="lib.fq.gz"):
        d = os.path.join(root, name.replace(" ", "_"))
        os.makedirs(d)
        with open(os.path.join(d, name_gz), "wb") as fh:
            fh.write(data if isinstance(data, bytes) and data[:2] == b"\x1f\x8b" else bgzf_compress(data, block=BLOCK))
        for mode in modes:
            exp = expected[mode] if isinstance(expected, dict) else expected
            cases[name, mode] = (d, {name_gz: [BARCODES, SAMPLES]}, tags, maxreads, inject, env or {}, exp)

    data = text.encode("utf-8")
    add("lf", data, "sharded")
    add("crlf", text.replace("\n", "\r\n").encode("utf-8"), "sharded")
    add("maxreads in rank 1", data, "sharded", maxreads=n * 11 // 20)
    mixed = list(recs)
    for i in range(n * 11 // 20, n * 12 // 20, 7):               # valid non-ASCII in rank 1's range
        c1, s, c2, q = mixed[i].split("\n")[:4]
        mixed[i] = "\n".join([c1, s[:20] + "é" + s[20:], c2, q]) + "\n"
    uni = "".join(mixed).encode("utf-8")
    add("non-ascii", uni, {"plain": "fallback", "adapter": "sharded"})
    at = uni.index("é".encode("utf-8"))
    add("invalid utf-8", uni[:at] + b"\xff" + uni[at + 2:], "fallback", modes=("plain",))
    good = bgzf_compress(data, block=BLOCK)
    marks = [i for i in range(len(good)) if good.startswith(b"\x1f\x8b\x08\x04", i)]
    bad = bytearray(good)
    bad[marks[len(marks) * 11 // 20] + 40] ^= 0x10                # a flipped bit in a member of rank 1's range
    add("corrupt member", bytes(bad), "fallback")
    add("lone cr", text.replace("\n", "\r").encode("utf-8"), "fallback")
    giant = "".join(recs[:300]) + "@g\n" + "".join(rng.choice("ACGT") for _ in range(4 << 20)) + "\n+\n" + "".join(recs[-300:])
    add("giant line at the cuts", giant.encode("ascii"), "fallback")
    add("inflate fails on rank 1", data, "fallback", inject=True)
    add("bgzf then gzip", good[:-28] + gzip.compress(data[:5000]), "dealt")
    add("gzip", gzip.compress(data), "dealt")
    add("TDG_GZDEV=0", data, "dealt", env={"TDG_GZDEV": "0"})
    return cases


def _rank_main(rank, world, port, cases, out_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    counting.SHARD_MIN_BYTES = 1024
    counting.HEAD_CAP = HEAD_CAP
    counting.LOOKAHEAD_CAP = LOOKAHEAD_CAP

    def cpu_reduce(ptr, rows, cols, eng):
        t = torch.from_numpy(eng.read_matrix())
        dist.all_reduce(t)
        a = np.ascontiguousarray(t.numpy())
        eng.memcpy_h2d(ptr, a.ctypes.data, a.nbytes)

    def no_reduce(ptr, rows, cols, eng):         # rank 0 raised before its reduce: no collective to meet
        pass

    def fail(*args, **kw):
        raise _native.TdgError(_native.TDG_ERR_NOMEM, "injected failure")

    results = {}
    for (name, mode), (d, key, tags, maxreads, inject, env, _exp) in sorted(cases.items()):
        os.chdir(d)
        with pytest.MonkeyPatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            if rank == 1 and inject:
                mp.setattr(_native.Engine, "bgzf_inflate_device", fail)
            results[name, mode] = _run(mode, key, tags, "TGCAG", "PstI-MspI-Hall", maxreads, rank=rank, world=world,
                                       reduce=no_reduce if name in RAISES else cpu_reduce, gather=counting.dist_gather)
    with open(os.path.join(out_dir, "rank%d.pkl" % rank), "wb") as fh:
        pickle.dump(results, fh)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_bgzf_count_equals_one_rank(world, tmp_path, library, monkeypatch):
    import torch.multiprocessing as mp
    cases = _cases(str(tmp_path), library)
    want = {}
    old = os.getcwd()
    try:
        for case, (d, key, tags, maxreads, _inject, env, exp) in cases.items():
            os.chdir(d)
            with monkeypatch.context() as m:
                for k, v in env.items():
                    m.setenv(k, v)
                want[case] = _run(case[1], key, tags, "TGCAG", "PstI-MspI-Hall", maxreads)
                m.setattr(counting, "SHARD_MIN_BYTES", 1024)
                assert bool(counting.shard_files(sorted(key), world)) == (exp != "dealt"), case
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
        expected = cases[case][6]
        if name in RAISES:
            assert res is None and err is not None, (case, res)
            if name == "invalid utf-8":
                assert err[0] == "UnicodeDecodeError", err
            assert got[0][case][2] == err, (case, got[0][case][2])
            assert got[0][case][1] == out, case
            for r in range(1, world):                           # as when the file is dealt whole to rank 0
                g_res, g_out, g_err = got[r][case]
                assert g_err is None and g_res[2] == {} and g_out == "", (case, r, g_err)
            continue
        assert err is None, (case, err)
        for r in range(world):
            g_res, g_out, g_err = got[r][case]
            assert g_err is None, (case, r, g_err)
            assert g_res[0] == res[0] and g_res[1] == res[1], (case, r)
            for f, t in g_res[2].items():
                assert t == res[2][f], (case, r, f)
        holders = [sorted(got[r][case][0][2]) for r in range(world)]
        f = sorted(res[2])
        assert holders == ([f] * world if expected == "sharded" else [f] + [[]] * (world - 1)), (case, holders)
        assert got[0][case][1] == out, case
        assert all(got[r][case][1] == "" for r in range(1, world)), case
