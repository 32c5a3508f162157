"""Reading BGZF files back for the tests: the member framing (SAMv1 4.1) and the dynamic-Huffman block
header of RFC 1951 3.2.7, with the rules every decoder of the project enforces."""

import struct
import zlib

BLOCK = 65280
EOF_MEMBER = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
CL_ORDER = (16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15)


def members(blob):
    """Split a BGZF file into members, checking every header field; returns [(member bytes, text)]."""
    out = []
    p = 0
    while p < len(blob):
        assert blob[p:p + 4] == b"\x1f\x8b\x08\x04", "ID1 ID2 CM FLG at %d" % p
        xlen, = struct.unpack_from("<H", blob, p + 10)
        assert xlen == 6 and blob[p + 12:p + 16] == b"BC\x02\x00", "BC extra field at %d" % p
        bsize, = struct.unpack_from("<H", blob, p + 16)
        size = bsize + 1
        assert size <= 65536
        m = blob[p:p + size]
        assert len(m) == size
        d = zlib.decompressobj(-15)
        text = d.decompress(m[18:-8]) + d.flush()
        assert d.eof and not d.unused_data, "the deflate stream fills the member exactly"
        crc, isize = struct.unpack_from("<II", m, size - 8)
        assert crc == zlib.crc32(text) and isize == len(text)
        out.append((m, text))
        p += size
    return out


def check_file(blob, want):
    """blob is a BGZF file of want: members of 65,280-byte cuts, then the EOF member."""
    ms = members(blob)
    assert ms and ms[-1][0] == EOF_MEMBER
    texts = [t for _, t in ms[:-1]]
    assert all(len(t) == BLOCK for t in texts[:-1]) and all(texts)
    for k, t in enumerate(texts):
        assert t == want[k * BLOCK:(k + 1) * BLOCK], "member %d" % k
    assert len(texts) == (len(want) + BLOCK - 1) // BLOCK
    return ms


class _Bits:
    def __init__(self, data):
        self.v = int.from_bytes(data, "little")
        self.p = 0

    def get(self, n):
        x = (self.v >> self.p) & ((1 << n) - 1)
        self.p += n
        return x


def _kraft_complete(lens):
    return sum(2.0 ** (15 - ln) for ln in lens if ln) == 2.0 ** 15


def _decode_canonical(lens):
    """{(length, bit-reversed code): symbol}"""
    table, code = {}, 0
    for ln in range(1, 16):
        for s, l in enumerate(lens):
            if l == ln:
                rev = int(format(code, "0%db" % ln)[::-1], 2)
                table[(ln, rev)] = s
                code += 1
        code <<= 1
    return table


def block_header(deflate):
    """The rules checked on the first block of a deflate stream; returns (BTYPE, HLIT, HDIST, HCLEN)."""
    b = _Bits(deflate)
    b.get(1)
    btype = b.get(2)
    if btype != 2:
        return btype, None, None, None
    hlit, hdist, hclen = b.get(5) + 257, b.get(5) + 1, b.get(4) + 4
    assert hlit <= 286 and hdist <= 30 and hclen <= 19          # never symbols 286/287, distances 30/31
    cl = [0] * 19
    for i in range(hclen):
        cl[CL_ORDER[i]] = b.get(3)
    assert sum(1 for x in cl if x) >= 2 and _kraft_complete(cl), cl
    table = _decode_canonical(cl)
    seq = []

    def sym():
        code, ln = 0, 0
        while True:
            code |= b.get(1) << ln
            ln += 1
            if (ln, code) in table:
                return table[(ln, code)]
            assert ln < 8

    for part in (hlit, hdist):
        lens = []
        while len(lens) < part:
            s = sym()
            if s < 16:
                lens.append(s)
            elif s == 16:
                assert lens, "repeat code 16 first"
                lens += [lens[-1]] * (3 + b.get(2))
            elif s == 17:
                lens += [0] * (3 + b.get(3))
            else:
                lens += [0] * (11 + b.get(7))
        assert len(lens) == part, "a run crosses from the literal/length lengths into the distance lengths"
        seq.append(lens)
    lit, dist = seq
    for lens in (lit, dist):
        assert sum(1 for x in lens if x) >= 2 and max(lens) <= 15 and _kraft_complete(lens)
    assert lit[256], "end of block has a code"
    return btype, hlit, hdist, hclen
