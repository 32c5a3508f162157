"""ctypes wrapper of the CPU harness over the splitter's BGZF encoder
(tests/native/bgzf_check.cpp; product code: tagdigger_b200/csrc/tdg_bgzf.cuh)."""

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "native", "bgzf_check.cpp")
_LIB = os.path.join(_HERE, "native", "libbgzf_check.so")
_DEPS = [os.path.join(os.path.dirname(_HERE), "tagdigger_b200", "csrc", "tdg_bgzf.cuh")]

BLOCK = 65280
_lib = None


def build(force=False):
    if not force and os.path.exists(_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(_LIB) for d in [_SRC] + _DEPS):
        return _LIB
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", _LIB, _SRC, "-lz"])
    return _LIB


def _L():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        L.bzc_huff_lengths.restype = ctypes.c_int
        L.bzc_huff_lengths.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
        L.bzc_member.restype = ctypes.c_longlong
        L.bzc_member.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib = L
    return _lib


def huff_lengths(freq, maxbits):
    """(code lengths, frequencies as the encoder left them) for a histogram."""
    f = np.ascontiguousarray(freq, dtype=np.uint32).copy()
    ln = np.zeros(len(f), dtype=np.uint8)
    _L().bzc_huff_lengths(f.ctypes.data, len(f), maxbits, ln.ctypes.data)
    return ln, f


def member(data, matches=None):
    """(one BGZF member for data (<= 65,280 bytes), dynamic block?).  matches: per-position uint32
    array (len << 16 | (dist - 1), 0 = literal) used instead of the encoder's own match search."""
    data = bytes(data)
    out = np.zeros(len(data) + 64, dtype=np.uint8)
    info = np.zeros(1, dtype=np.uint32)
    m = None
    if matches is not None:
        m = np.ascontiguousarray(matches, dtype=np.uint32)
        assert len(m) == len(data)
    n = _L().bzc_member(data, len(data), m.ctypes.data if m is not None else None, out.ctypes.data, info.ctypes.data)
    assert n > 0
    return out[:n].tobytes(), bool(info[0])


def compress(data):
    """A whole BGZF file: members of 65,280-byte cuts, then the end-of-file member."""
    data = bytes(data)
    return b"".join(member(data[k:k + BLOCK])[0] for k in range(0, len(data), BLOCK)) + member(b"")[0]
