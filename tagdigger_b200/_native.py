"""Build and ctypes binding of ``libtagdigger_b200.so`` (include/tagdigger_b200.h).

The library is compiled in-tree with nvcc for sm_100a only.  There is no CPU
counting path: every ``Engine`` method that counts reads ends in the CUDA kernel
of ``csrc/tdg_kernel.cuh``, and constructing an ``Engine`` without a CUDA device
(or without the built library) raises.
"""

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_PATH = os.environ.get("TDG_LIB") or os.path.join(_HERE, "libtagdigger_b200.so")   # TDG_LIB: tuning builds (scripts/sweep.py)
_SOURCES = ["tdg_api.cu", "tdg_text.h", "tdg_comm.h", "tdg_kernel.cuh", "tdg_match.h", "tdg_tables.h", "tdg_trim.cuh", "tdg_split.cuh", "tdg_feed.h", "tdg_pgz.h", "tdg_csv.h",
            "tdg_gzlane.h", "tdg_gzchain.h", "tdg_gzdev.cuh", "tdg_gzfeed.cuh", "tdg_pool.h", "tdg_bgzf.cuh"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-diag-suppress", "20014,20011", "-shared"]

ABI_VERSION = 2            # include/tagdigger_b200.h: TDG_ABI_VERSION
TDG_OK = 0
TDG_ERR_CUDA, TDG_ERR_ARG, TDG_ERR_IO, TDG_ERR_STATE, TDG_ERR_NOMEM, TDG_ERR_GZIP, TDG_ERR_UTF8 = -1, -2, -3, -4, -5, -6, -7
TDG_ANY_BASE = 1
TDG_PREV_NONE, TDG_PREV_LF, TDG_PREV_CR, TDG_PREV_OTHER = 0, 1, 2, 3
TDG_LINE_CHAINED = (1 << 64) - 1
TDG_TILE_BYTES = 16384
TDG_HALO_BYTES = 512
NO_LIMIT = (1 << 63)

EXPORTS = """tdg_abi_version tdg_create tdg_destroy tdg_last_error tdg_set_tags tdg_set_matrix
tdg_bind_matrix tdg_zero_matrix tdg_begin_file tdg_reset_file tdg_submit tdg_end_file tdg_count_device
tdg_count_lines_device tdg_count_file tdg_count_file2 tdg_last_file_info tdg_gz_inflate_host tdg_release_scratch tdg_sync tdg_file_totals tdg_read_matrix tdg_matrix_min tdg_comm_unique_id tdg_comm_init tdg_allreduce_matrix tdg_finish
tdg_matrix_device_ptr tdg_stream tdg_stream_wait tdg_other_stream_wait tdg_host_alloc
tdg_host_free tdg_device_alloc tdg_device_free tdg_memcpy_h2d tdg_memcpy_d2h tdg_launch_count
tdg_timing_begin tdg_timing_end tdg_set_trim tdg_trim_batch tdg_split_batch tdg_split_begin tdg_split_block
tdg_split_count_begin tdg_split_count_block tdg_split_count_batch tdg_split_bgzf tdg_bgzf_append tdg_bgzf_finish tdg_feed_open tdg_feed_read tdg_feed_close tdg_match_batch tdg_write_counts_csv tdg_write_geno_csv""".split()


class TdgError(RuntimeError):
    def __init__(self, code, message):
        RuntimeError.__init__(self, "tagdigger_b200 error %d: %s" % (code, message))
        self.code = code
        self.message = message


def _stale():
    if os.environ.get("TDG_LIB"):
        return False
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    srcs = [os.path.join(_CSRC, s) for s in _SOURCES] + [os.path.join(_INCLUDE, "tagdigger_b200.h")]
    return any(os.path.exists(s) and os.path.getmtime(s) > t for s in srcs)


def build(force=False, verbose=False):
    """Compile csrc/ into libtagdigger_b200.so with nvcc (cross-compiles without a GPU)."""
    if not force and not _stale():
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB_PATH, os.path.join(_CSRC, "tdg_api.cu"), "-lz"]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, universal_newlines=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout)
    if verbose:
        print(proc.stdout)
    return LIB_PATH


_lib = None


def lib():
    """The loaded library.  Builds it when sources are newer and nvcc exists;
    raises if it is neither built nor buildable (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if _stale():
        try:
            build()
        except (OSError, RuntimeError) as e:
            if not os.path.exists(LIB_PATH):
                raise
            import warnings
            warnings.warn("tagdigger_b200: the sources are newer than %s and rebuilding failed (%s); loading the "
                          "existing library -- its ABI version is checked below" % (LIB_PATH, str(e)[:200]), RuntimeWarning)
    L = ctypes.CDLL(LIB_PATH)
    L.tdg_abi_version.restype = ctypes.c_int
    if L.tdg_abi_version() != ABI_VERSION:
        raise RuntimeError("%s has ABI version %d, this package needs %d: rebuild it (python -c 'import "
                           "__graft_entry__ as g; g.build()')" % (LIB_PATH, L.tdg_abi_version(), ABI_VERSION))
    vp, u64, u32, i32, sz = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_size_t
    sig = {
        "tdg_abi_version": (i32, []),
        "tdg_create": (i32, [ctypes.POINTER(vp), i32, sz]),
        "tdg_destroy": (None, [vp]),
        "tdg_last_error": (ctypes.c_char_p, [vp]),
        "tdg_set_tags": (i32, [vp, vp, vp, vp, u32, u32]),
        "tdg_set_matrix": (i32, [vp, u32, u32]),
        "tdg_bind_matrix": (i32, [vp, vp, u32, u32]),
        "tdg_zero_matrix": (i32, [vp]),
        "tdg_begin_file": (i32, [vp, vp, vp, vp, vp, u32, u32]),
        "tdg_reset_file": (i32, [vp]),
        "tdg_submit": (i32, [vp, vp, sz, u64]),
        "tdg_end_file": (i32, [vp, u64]),
        "tdg_count_device": (i32, [vp, vp, sz, u64, i32, u64]),
        "tdg_count_lines_device": (i32, [vp, vp, sz, u64, i32, vp]),
        "tdg_count_file": (i32, [vp, ctypes.c_char_p, i32, u64, vp]),
        "tdg_count_file2": (i32, [vp, ctypes.c_char_p, i32, u64, vp, ctypes.c_char_p, i32]),
        "tdg_gz_inflate_host": (i32, [vp, ctypes.c_char_p, vp, sz, vp, vp, vp]),
        "tdg_last_file_info": (i32, [vp, vp]),
        "tdg_release_scratch": (i32, [vp]),
        "tdg_sync": (i32, [vp]),
        "tdg_file_totals": (i32, [vp, vp]),
        "tdg_read_matrix": (i32, [vp, vp]),
        "tdg_matrix_min": (i32, [vp, vp]),
        "tdg_comm_unique_id": (i32, [vp]),
        "tdg_comm_init": (i32, [vp, vp, i32, i32]),
        "tdg_allreduce_matrix": (i32, [vp]),
        "tdg_finish": (i32, [vp, vp, vp]),
        "tdg_matrix_device_ptr": (vp, [vp]),
        "tdg_stream": (vp, [vp]),
        "tdg_stream_wait": (i32, [vp, vp]),
        "tdg_other_stream_wait": (i32, [vp, vp]),
        "tdg_host_alloc": (vp, [vp, sz]),
        "tdg_host_free": (None, [vp, vp]),
        "tdg_device_alloc": (vp, [vp, sz]),
        "tdg_device_free": (None, [vp, vp]),
        "tdg_memcpy_h2d": (i32, [vp, vp, vp, sz]),
        "tdg_memcpy_d2h": (i32, [vp, vp, vp, sz]),
        "tdg_launch_count": (u64, [vp]),
        "tdg_timing_begin": (i32, [vp]),
        "tdg_timing_end": (i32, [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(u32)]),
        "tdg_set_trim": (i32, [vp, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, u32, vp, vp, vp, vp, vp, vp]),
        "tdg_trim_batch": (i32, [vp, vp, vp, vp, vp, u32, vp]),
        "tdg_split_batch": (i32, [vp, vp, vp, u32, vp, u32, u32, vp, vp]),
        "tdg_split_begin": (i32, [vp, vp, vp, u32, u32]),
        "tdg_split_block": (i32, [vp, vp, sz, i32, u64, ctypes.POINTER(u64), ctypes.POINTER(u64), ctypes.POINTER(i32),
                                  ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp)]),
        "tdg_split_count_begin": (i32, [vp, vp, vp, vp, u32, u32, vp]),
        "tdg_split_count_block": (i32, [vp, vp, sz, i32, u64, ctypes.POINTER(u64), ctypes.POINTER(u64), ctypes.POINTER(i32), vp]),
        "tdg_split_count_batch": (i32, [vp, vp, vp, vp, u32, vp]),
        "tdg_split_bgzf": (i32, [vp, i32]),
        "tdg_bgzf_append": (i32, [vp, vp, vp, ctypes.POINTER(vp), ctypes.POINTER(vp)]),
        "tdg_bgzf_finish": (i32, [vp, ctypes.POINTER(vp), ctypes.POINTER(vp)]),
        "tdg_feed_open": (i32, [ctypes.POINTER(vp), ctypes.c_char_p, i32]),
        "tdg_feed_read": (ctypes.c_longlong, [vp, vp, sz]),
        "tdg_feed_close": (None, [vp]),
        "tdg_match_batch": (i32, [vp, vp, vp, u32, vp, vp]),
        "tdg_write_counts_csv": (i32, [ctypes.c_char_p, vp, u32, u32, ctypes.c_char_p, sz, ctypes.c_char_p, vp, i32]),
        "tdg_write_geno_csv": (i32, [ctypes.c_char_p, vp, u32, u32, vp, vp, u32, ctypes.c_char_p, sz, ctypes.c_char_p, vp, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _csr(seqs, offset_dtype):
    blob = "".join(seqs).encode("ascii")
    off = np.zeros(len(seqs) + 1, dtype=offset_dtype)
    if len(seqs):
        np.cumsum([len(s) for s in seqs], out=off[1:])
    return blob, off


def limit_from_maxreads(maxreads):
    """The reference checks ``readscount >= maxreads`` after each read
    (tagdigger_fun.py:272-273): at least one read is processed, and a
    fractional maxreads rounds up."""
    if maxreads is None:
        return NO_LIMIT
    m = float(maxreads)
    if m != m:                       # NaN never compares >=
        return NO_LIMIT
    if m >= float(NO_LIMIT):
        return NO_LIMIT
    lim = int(m)
    if lim < m:
        lim += 1
    return max(1, lim)


def _csv_line(fields):
    """One row as Python's csv.writer (default dialect) writes it, as bytes."""
    import csv
    import io
    buf = io.StringIO(newline="")
    csv.writer(buf).writerow(fields)
    return buf.getvalue().encode("utf-8")


def _csv_labels(names):
    """CSV-escaped first fields of rows that have more fields after them."""
    out = []
    for n in names:
        line = _csv_line([n, "x"])
        out.append(line[:-len(b",x\r\n")])
    blob = b"".join(out)
    off = np.zeros(len(out) + 1, dtype=np.uint64)
    if out:
        np.cumsum([len(x) for x in out], out=off[1:])
    return blob, off


def write_counts_csv(path, matrix, samnames, tagnames, threads=8):
    """writeCounts for an int32 ndarray [samples x tags]: native, multithreaded, byte-identical."""
    m = np.ascontiguousarray(matrix, dtype=np.int32)
    header = _csv_line([""] + list(tagnames))
    blob, off = _csv_labels(samnames)
    L = lib()
    rc = L.tdg_write_counts_csv(os.fsencode(path), m.ctypes.data, m.shape[0], m.shape[1] if m.ndim == 2 else 0,
                                header, len(header), blob, off.ctypes.data, threads)
    if rc != TDG_OK:
        raise OSError(L.tdg_last_error(None).decode())


def write_geno_csv(path, matrix, samnames, markers, col0, col1, threads=8):
    """writeDiploidGeno for an int32 ndarray: marker m is called from columns col0[m], col1[m]."""
    m = np.ascontiguousarray(matrix, dtype=np.int32)
    header = _csv_line([""] + list(markers))
    blob, off = _csv_labels(samnames)
    c0 = np.asarray(col0, dtype=np.uint32)
    c1 = np.asarray(col1, dtype=np.uint32)
    L = lib()
    rc = L.tdg_write_geno_csv(os.fsencode(path), m.ctypes.data, m.shape[0], m.shape[1] if m.ndim == 2 else 0,
                              c0.ctypes.data, c1.ctypes.data, len(c0), header, len(header), blob, off.ctypes.data, threads)
    if rc != TDG_OK:
        raise OSError(L.tdg_last_error(None).decode())


class Engine(object):
    """One context = one CUDA device (include/tagdigger_b200.h)."""

    def __init__(self, device=0, chunk_bytes=0):
        self._L = lib()
        self._h = ctypes.c_void_p()
        rc = self._L.tdg_create(ctypes.byref(self._h), device, chunk_bytes)
        if rc != TDG_OK:
            msg = self._L.tdg_last_error(None).decode()
            self._h = ctypes.c_void_p()
            raise TdgError(rc, msg)
        self.device = device
        self.rows = self.cols = 0

    # -- plumbing ----------------------------------------------------------
    def _ck(self, rc):
        if rc != TDG_OK:
            raise TdgError(rc, self._L.tdg_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.tdg_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:      # noqa: BLE001 - interpreter shutdown
            pass

    # -- tables ------------------------------------------------------------
    def set_tags(self, seqs, cols=None, any_base=False):
        """seqs: the effective (prefix-free) tag list; cols[i]: matrix column."""
        if cols is None:
            cols = range(len(seqs))
        blob, off = _csr(seqs, np.uint64)
        col = np.asarray(list(cols), dtype=np.int32)
        self._keep_tags = (blob, off, col)
        self._ck(self._L.tdg_set_tags(self._h, blob, off.ctypes.data, col.ctypes.data, len(seqs),
                                      TDG_ANY_BASE if any_base else 0))

    def set_matrix(self, rows, cols):
        self._ck(self._L.tdg_set_matrix(self._h, rows, cols))
        self.rows, self.cols = rows, cols
        self._hits = 0

    def bind_matrix(self, dev_ptr, rows, cols):
        self._ck(self._L.tdg_bind_matrix(self._h, dev_ptr, rows, cols))
        self.rows, self.cols = rows, cols

    def zero_matrix(self):
        self._ck(self._L.tdg_zero_matrix(self._h))
        self._hits = 0

    def begin_file(self, patterns, rows, tag_offs, any_base=False):
        blob, off = _csr(patterns, np.uint32)
        row = np.asarray(list(rows), dtype=np.int32)
        toff = np.asarray(list(tag_offs), dtype=np.uint32)
        self._ck(self._L.tdg_begin_file(self._h, blob, off.ctypes.data, row.ctypes.data, toff.ctypes.data,
                                        len(patterns), TDG_ANY_BASE if any_base else 0))

    def reset_file(self):
        self._ck(self._L.tdg_reset_file(self._h))

    # -- counting ----------------------------------------------------------
    def submit(self, data, reads_limit=NO_LIMIT):
        """data: bytes / bytearray / uint8 ndarray / (address, nbytes)."""
        if isinstance(data, tuple):
            addr, n = data
        elif isinstance(data, np.ndarray):
            addr, n = data.ctypes.data, data.nbytes
            self._pin = data
        else:
            buf = np.frombuffer(data, dtype=np.uint8)
            addr, n = buf.ctypes.data, buf.nbytes
            self._pin = buf
        self._ck(self._L.tdg_submit(self._h, addr, n, reads_limit))

    def end_file(self, reads_limit=NO_LIMIT):
        self._ck(self._L.tdg_end_file(self._h, reads_limit))

    def count_device(self, dev_ptr, n, line_base=0, prev_kind=TDG_PREV_NONE, reads_limit=NO_LIMIT):
        self._ck(self._L.tdg_count_device(self._h, dev_ptr, n, line_base, prev_kind, reads_limit))

    def count_lines_device(self, dev_ptr, n, line_base=0, prev_kind=TDG_PREV_NONE):
        st = np.zeros(2, dtype=np.uint64)
        self._ck(self._L.tdg_count_lines_device(self._h, dev_ptr, n, line_base, prev_kind, st.ctypes.data))
        return int(st[0]), int(st[1])

    def count_file(self, path, gz, reads_limit=NO_LIMIT, next_path=None, next_gz=False):
        """next_path: the file that will be counted after this one (its reading starts now)."""
        tot = np.zeros(4, dtype=np.uint64)
        self._ck(self._L.tdg_count_file2(self._h, os.fsencode(path), 1 if gz else 0, reads_limit, tot.ctypes.data,
                                         os.fsencode(next_path) if next_path else None, 1 if next_gz else 0))
        self.note_hits(int(tot[2]))
        return [int(x) for x in tot]

    def gz_inflate_host(self, path, cap):
        """The gzip feed of count_file by itself (tdg_gz_inflate_host): (bytes, info, ms) with info =
        {rounds, chunks, accepted, mode} -- mode 0 all on the device, 1 host parallel reader resumed,
        2 zlib resumed, -1 not taken by the device feed -- and ms = milliseconds per stage."""
        out = np.empty(cap, dtype=np.uint8)
        n = ctypes.c_uint64(0)
        info = np.zeros(4, dtype=np.int64)
        ms = np.zeros(6, dtype=np.float64)
        self._ck(self._L.tdg_gz_inflate_host(self._h, os.fsencode(path), out.ctypes.data, cap, ctypes.byref(n), info.ctypes.data,
                                             ms.ctypes.data))
        keys = ("upload", "scan", "decode", "resolve", "crc", "copy")
        return (out[:n.value].tobytes(), {"rounds": int(info[0]), "chunks": int(info[1]), "accepted": int(info[2]), "mode": int(info[3])},
                dict(zip(keys, (round(float(x), 2) for x in ms))))

    def last_file_info(self):
        """How the last count_file fed its file: {rounds, accepted, mode} (mode 0 device, 1 host took over, -1 host only)."""
        info = np.zeros(3, dtype=np.int64)
        self._ck(self._L.tdg_last_file_info(self._h, info.ctypes.data))
        return {"rounds": int(info[0]), "accepted": int(info[1]), "mode": int(info[2])}

    def release_scratch(self):
        """Free the working buffers of the device-side gzip feed (kept between files otherwise)."""
        self._ck(self._L.tdg_release_scratch(self._h))

    def sync(self):
        self._ck(self._L.tdg_sync(self._h))

    def file_totals(self):
        tot = np.zeros(4, dtype=np.uint64)
        self._ck(self._L.tdg_file_totals(self._h, tot.ctypes.data))
        return [int(x) for x in tot]

    def note_hits(self, hits):
        """Overflow guard (cells are int32, the reference's counts are unbounded Python ints):
        ``hits`` more reads were counted since the last check.  While fewer than 2**31 reads have
        been counted into the matrix no cell can have wrapped; beyond that the smallest cell is
        looked at (a wrapped cell is negative) and OverflowError raised."""
        self._hits = getattr(self, "_hits", 0) + int(hits)
        if self._hits >= (1 << 31):
            m = ctypes.c_int32(0)
            self._ck(self._L.tdg_matrix_min(self._h, ctypes.byref(m)))
            if m.value < 0 or int(hits) >= (1 << 32):
                raise OverflowError("a count passed 2**31 - 1: the device matrix holds int32 cells "
                                    "(the reference counts with unbounded integers); split the key")

    # -- multi-GPU ---------------------------------------------------------
    @staticmethod
    def comm_unique_id():
        """128-byte NCCL id made by rank 0 (hand it to every rank, then comm_init everywhere)."""
        buf = ctypes.create_string_buffer(128)
        rc = lib().tdg_comm_unique_id(buf)
        if rc != TDG_OK:
            raise TdgError(rc, lib().tdg_last_error(None).decode())
        return buf.raw

    def comm_init(self, unique_id, nranks, rank):
        self._ck(self._L.tdg_comm_init(self._h, ctypes.c_char_p(unique_id), nranks, rank))

    def allreduce_matrix(self):
        """Sum the count matrices of all ranks in place (one ncclAllReduce on the engine's stream)."""
        self._ck(self._L.tdg_allreduce_matrix(self._h))

    def read_matrix(self, out=None):
        if out is None:
            out = np.empty((self.rows, self.cols), dtype=np.int32)
        self._ck(self._L.tdg_read_matrix(self._h, out.ctypes.data))
        return out

    # -- memory / streams --------------------------------------------------
    def matrix_ptr(self):
        return self._L.tdg_matrix_device_ptr(self._h)

    def stream(self):
        return self._L.tdg_stream(self._h)

    def stream_wait(self, other):
        self._ck(self._L.tdg_stream_wait(self._h, other))

    def other_stream_wait(self, other):
        self._ck(self._L.tdg_other_stream_wait(self._h, other))

    def host_alloc(self, n):
        p = self._L.tdg_host_alloc(self._h, n)
        if not p:
            raise TdgError(TDG_ERR_NOMEM, "pinned allocation of %d bytes failed" % n)
        return p

    def host_free(self, p):
        self._L.tdg_host_free(self._h, p)

    def device_alloc(self, n):
        p = self._L.tdg_device_alloc(self._h, n)
        if not p:
            raise TdgError(TDG_ERR_NOMEM, "device allocation of %d bytes failed" % n)
        return p

    def device_free(self, p):
        self._L.tdg_device_free(self._h, p)

    def memcpy_h2d(self, dev, host_addr, n):
        self._ck(self._L.tdg_memcpy_h2d(self._h, dev, host_addr, n))

    def memcpy_d2h(self, host_addr, dev, n):
        self._ck(self._L.tdg_memcpy_d2h(self._h, host_addr, dev, n))

    def upload(self, data):
        """Copy a host FASTQ image to a fresh, suitably padded device buffer.
        Returns (device pointer, nbytes); free with device_free."""
        arr = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
        n = arr.nbytes
        cap = (n + TDG_TILE_BYTES - 1) // TDG_TILE_BYTES * TDG_TILE_BYTES + TDG_HALO_BYTES
        p = self.device_alloc(cap)
        if n:
            self.memcpy_h2d(p, arr.ctypes.data, n)
        return p, n

    # -- accounting --------------------------------------------------------
    def launch_count(self):
        return int(self._L.tdg_launch_count(self._h))

    def timing_begin(self):
        self._ck(self._L.tdg_timing_begin(self._h))

    def timing_end(self):
        ms = ctypes.c_double(0)
        n = ctypes.c_uint32(0)
        self._ck(self._L.tdg_timing_end(self._h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    # -- trim decision ------------------------------------------------------
    def set_trim(self, site0, site1, a0, a1_list, cands):
        """cands[b]: list of (which, length, slice index) for barcode b (trimming.trim_tables)."""
        a1_blob, a1_off = _csr(a1_list, np.uint32)
        cand_off = np.zeros(len(cands) + 1, dtype=np.uint32)
        if len(cands):
            np.cumsum([len(c) for c in cands], out=cand_off[1:])
        flat = [t for c in cands for t in c]
        which = np.asarray([t[0] for t in flat], dtype=np.uint8)
        clen = np.asarray([t[1] for t in flat], dtype=np.uint16)
        cidx = np.asarray([t[2] for t in flat], dtype=np.int16)
        self._ck(self._L.tdg_set_trim(self._h, site0.encode("ascii"), site1.encode("ascii"), a0.encode("ascii"),
                                      len(cands), a1_blob, a1_off.ctypes.data, cand_off.ctypes.data,
                                      clen.ctypes.data, cidx.ctypes.data, which.ctypes.data))

    def trim_batch(self, seqs, bars, starts):
        """seqs: list of bytes/str sequence lines; returns the list of slice2 values."""
        raw = [x.encode("utf-8") if isinstance(x, str) else bytes(x) for x in seqs]
        blob = b"".join(raw)
        off = np.zeros(len(raw) + 1, dtype=np.uint64)
        if raw:
            np.cumsum([len(x) for x in raw], out=off[1:])
        bar = np.asarray(list(bars), dtype=np.int32)
        start = np.asarray(list(starts), dtype=np.uint32)
        out = np.empty(len(raw), dtype=np.int32)
        self._ck(self._L.tdg_trim_batch(self._h, blob, off.ctypes.data, bar.ctypes.data, start.ctypes.data,
                                        len(raw), out.ctypes.data))
        return [int(x) for x in out]

    def split_batch(self, seqs, bar_lens, cutlen):
        """seqs: list of stripped sequence lines (bytes/str).  Returns (barcode index or -1,
        slice2 or 999) arrays -- the two per-read decisions of barcodeSplitter."""
        raw = [x.encode("utf-8") if isinstance(x, str) else bytes(x) for x in seqs]
        blob = b"".join(raw)
        off = np.zeros(len(raw) + 1, dtype=np.uint64)
        if raw:
            np.cumsum([len(x) for x in raw], out=off[1:])
        blen = np.asarray(list(bar_lens), dtype=np.uint32)
        bar = np.empty(len(raw), dtype=np.int32)
        cut = np.empty(len(raw), dtype=np.int32)
        self._ck(self._L.tdg_split_batch(self._h, blob, off.ctypes.data, len(raw), blen.ctypes.data, len(blen),
                                         cutlen, bar.ctypes.data, cut.ctypes.data))
        return bar, cut

    def split_begin(self, barcodes, cutlen):
        """Barcode strings and cut-site length for split_block (after begin_file and set_trim)."""
        blob, off = _csr(list(barcodes), np.uint32)
        self._ck(self._L.tdg_split_begin(self._h, blob, off.ctypes.data, len(barcodes), cutlen))
        self._split_nbar = len(barcodes)

    def split_block(self, ptr, n, final, max_records):
        """One block of raw FASTQ bytes at host address ``ptr`` through the streaming splitter.
        Returns (records, consumed bytes, needs_host, pieces, flags): pieces[b] is a uint8 array
        (a view of pinned memory, valid until the next call) to append to barcode b's file,
        flags a uint8 array per record (1 barcode found | 2 clipped); both None when needs_host."""
        u64, vp = ctypes.c_uint64, ctypes.c_void_p
        nrec, used, host = u64(0), u64(0), ctypes.c_int(0)
        out, off, flags = vp(), vp(), vp()
        self._ck(self._L.tdg_split_block(self._h, ptr, n, 1 if final else 0, min(int(max_records), (1 << 64) - 1),
                                         ctypes.byref(nrec), ctypes.byref(used), ctypes.byref(host), ctypes.byref(out),
                                         ctypes.byref(off), ctypes.byref(flags)))
        if host.value or not out.value:
            return nrec.value, used.value, bool(host.value), None, None
        pieces = self._pieces(out, off)
        fl = np.ctypeslib.as_array(ctypes.cast(flags, ctypes.POINTER(ctypes.c_uint8)), shape=(max(nrec.value, 1),))[:nrec.value]
        return nrec.value, used.value, False, pieces, fl

    def split_count_begin(self, patterns, tag_offs, rows, any_base=False):
        """Count mode of the split started by split_begin (after set_tags and set_matrix): the
        stage-2 barcode+cutsite table (blank barcode: matchset.plan([''], tags, cutsite).bar with
        its tag offsets) and rows[b], the matrix row barcode b's reads are counted into."""
        blob, off = _csr(patterns, np.uint32)
        toff = np.asarray(list(tag_offs), dtype=np.uint32)
        row = np.asarray(list(rows), dtype=np.int32)
        if len(row) != self._split_nbar:
            raise ValueError("one row per barcode: %d given, %d barcodes" % (len(row), self._split_nbar))
        self._ck(self._L.tdg_split_count_begin(self._h, blob, off.ctypes.data, toff.ctypes.data, len(patterns),
                                               TDG_ANY_BASE if any_base else 0, row.ctypes.data))

    def split_count_block(self, ptr, n, final, max_records):
        """split_block that counts the trimmed reads into the matrix instead of returning them.
        Returns (records, consumed bytes, needs_host, totals): totals = [reads, with barcode and cut
        site, clipped on the 3' end, with tag] of the block; None when needs_host (nothing counted)."""
        u64 = ctypes.c_uint64
        nrec, used, host = u64(0), u64(0), ctypes.c_int(0)
        tot = np.zeros(4, dtype=np.uint64)
        self._ck(self._L.tdg_split_count_block(self._h, ptr, n, 1 if final else 0, min(int(max_records), (1 << 64) - 1),
                                               ctypes.byref(nrec), ctypes.byref(used), ctypes.byref(host), tot.ctypes.data))
        if host.value:
            return nrec.value, used.value, True, None
        self.note_hits(int(tot[3]))
        return nrec.value, used.value, False, [int(x) for x in tot]

    def split_count_batch(self, seqs, bars):
        """seqs: stage-2 lines t (stripped, upper case; bytes/str) of reads with barcode bars[i].
        Counts them into the matrix; returns the tag column of each, -1 = no tag."""
        raw = [x.encode("utf-8") if isinstance(x, str) else bytes(x) for x in seqs]
        blob = b"".join(raw)
        off = np.zeros(len(raw) + 1, dtype=np.uint64)
        if raw:
            np.cumsum([len(x) for x in raw], out=off[1:])
        bar = np.asarray(list(bars), dtype=np.int32)
        col = np.empty(len(raw), dtype=np.int32)
        self._ck(self._L.tdg_split_count_batch(self._h, blob, off.ctypes.data, bar.ctypes.data, len(raw), col.ctypes.data))
        self.note_hits(int(np.count_nonzero(col >= 0)))
        return col

    def _pieces(self, out, off):
        """Per-barcode views of out[off[b] .. off[b+1]) (pinned memory of the context)."""
        nbar = self._split_nbar
        offs = np.ctypeslib.as_array(ctypes.cast(off, ctypes.POINTER(ctypes.c_uint64)), shape=(nbar + 1,))
        total = int(offs[nbar])
        data = np.ctypeslib.as_array(ctypes.cast(out, ctypes.POINTER(ctypes.c_uint8)), shape=(max(total, 1),))
        return [data[int(offs[b]):int(offs[b + 1])] for b in range(nbar)]

    def split_bgzf(self, on):
        """BGZF output files for the split started by split_begin (empties every barcode's pending
        tail).  While on, split_block's pieces are completed BGZF members; bgzf_append takes the
        records written on the host, bgzf_finish ends the files."""
        self._ck(self._L.tdg_split_bgzf(self._h, 1 if on else 0))

    def bgzf_append(self, parts):
        """parts[b]: bytes appended to barcode b's uncompressed stream.  Returns the BGZF pieces to
        append to every barcode's file (views valid until the next call)."""
        if len(parts) != self._split_nbar:
            raise ValueError("one part per barcode: %d given, %d barcodes" % (len(parts), self._split_nbar))
        blob = b"".join(bytes(p) for p in parts)
        off = np.zeros(self._split_nbar + 1, dtype=np.uint64)
        np.cumsum([len(p) for p in parts], out=off[1:])
        out, o = ctypes.c_void_p(), ctypes.c_void_p()
        self._ck(self._L.tdg_bgzf_append(self._h, blob, off.ctypes.data, ctypes.byref(out), ctypes.byref(o)))
        return self._pieces(out, o)

    def bgzf_finish(self):
        """The last member of every barcode's file and the BGZF end-of-file member."""
        out, o = ctypes.c_void_p(), ctypes.c_void_p()
        self._ck(self._L.tdg_bgzf_finish(self._h, ctypes.byref(out), ctypes.byref(o)))
        return self._pieces(out, o)

    def match_batch(self, seqs):
        """seqs: list of stripped sequence lines (bytes/str).  Returns (row, col) arrays, -1 = no match."""
        raw = [x.encode("utf-8") if isinstance(x, str) else bytes(x) for x in seqs]
        blob = b"".join(raw)
        off = np.zeros(len(raw) + 1, dtype=np.uint64)
        if raw:
            np.cumsum([len(x) for x in raw], out=off[1:])
        row = np.empty(len(raw), dtype=np.int32)
        col = np.empty(len(raw), dtype=np.int32)
        self._ck(self._L.tdg_match_batch(self._h, blob, off.ctypes.data, len(raw), row.ctypes.data, col.ctypes.data))
        return row, col


class Feed:
    """The host feed on its own (csrc/tdg_feed.h): uncompressed bytes of a plain, gzip or BGZF
    file, read / inflated by host threads straight into caller memory."""

    def __init__(self, path, gz):
        self._L = lib()
        self._h = ctypes.c_void_p()
        rc = self._L.tdg_feed_open(ctypes.byref(self._h), os.fsencode(path), 1 if gz else 0)
        if rc != TDG_OK:
            raise TdgError(rc, self._L.tdg_last_error(None).decode())

    def read_into(self, ptr, cap):
        """Up to ``cap`` bytes to host address ``ptr``; 0 at the end of the file."""
        r = self._L.tdg_feed_read(self._h, ptr, cap)
        if r < 0:
            raise TdgError(int(r), self._L.tdg_last_error(None).decode())
        return int(r)

    def close(self):
        if self._h.value:
            self._L.tdg_feed_close(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
