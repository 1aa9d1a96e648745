"""Compressed blastouts: which reader a file needs, and the member table of a BGZF file.

The suffix decides, as the reference's `try_open` (waafle/utils.py) does: `.gz` is gzip, `.bz2` is bzip2, anything else
is text.  A `.gz` file is BGZF -- the gzip variant bgzip (htslib) writes -- when every member carries the `BC` extra
subfield and the chain of BSIZE values ends exactly at the end of the file.  Its member table then gives every member's
raw DEFLATE payload, ISIZE, CRC-32 and output offset from the headers alone, so the members can be inflated
independently on the GPU (csrc/wfl_inflate.cu).  Any header that does not follow the format makes the file generic
gzip, which the host inflates.
"""

import gzip
import struct

import numpy as np

TEXT, GZIP, BZIP2, BGZF = "text", "gzip", "bzip2", "bgzf"
# member table columns
PAYLOAD_OFF, PAYLOAD_LEN, ISIZE, CRC, OUT_OFF = range(5)
MAX_ISIZE = 65536
_HEAD = b"\x1f\x8b\x08\x04"   # gzip magic, deflate, FLG = FEXTRA only (what bgzip writes)


def suffix_kind(path):
    if path.endswith(".gz"):
        return GZIP
    if path.endswith(".bz2"):
        return BZIP2
    return TEXT


def bgzf_members(buf):
    """[n_members, 5] int64 member table of BGZF bytes `buf`, or None when `buf` is not BGZF.  Reads headers and
    trailers only (O(members)); nothing is decoded."""
    n, pos, out, rows = len(buf), 0, 0, []
    while pos < n:
        if n - pos < 28 or bytes(buf[pos:pos + 4]) != _HEAD:
            return None
        xlen = struct.unpack_from("<H", buf, pos + 10)[0]
        q, end, bsize = pos + 12, pos + 12 + xlen, None
        if end > n:
            return None
        while q + 4 <= end:
            slen = struct.unpack_from("<H", buf, q + 2)[0]
            if q + 4 + slen > end:
                return None
            if buf[q] == 66 and buf[q + 1] == 67 and slen == 2:   # "BC"
                if bsize is not None:
                    return None
                bsize = struct.unpack_from("<H", buf, q + 4)[0]
            q += 4 + slen
        if q != end or bsize is None:
            return None
        total = bsize + 1
        plen = total - 12 - xlen - 8
        if plen < 0 or pos + total > n:
            return None
        crc, isize = struct.unpack_from("<II", buf, pos + total - 8)
        # DEFLATE expands at most 1032:1; a larger claim cannot be a valid member (and would size the text buffer)
        if isize > MAX_ISIZE or isize > 1032 * plen + 1024:
            return None
        rows.append((end, plen, isize, crc, out))
        out += isize
        pos += total
    return np.array(rows, dtype=np.int64).reshape(-1, 5) if rows else None


def classify(path):
    """(kind, member table): (BGZF, table) for a BGZF `.gz`, (GZIP | BZIP2 | TEXT, None) otherwise."""
    kind = suffix_kind(path)
    if kind != GZIP:
        return kind, None
    import mmap
    with open(path, "rb") as fh:
        try:
            mm = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)
        except ValueError:   # an empty file
            return GZIP, None
        with mm:
            members = bgzf_members(mm)
    return (BGZF, members) if members is not None else (GZIP, None)


def text_size(members):
    return int(members[-1, OUT_OFF] + members[-1, ISIZE]) if len(members) else 0


def member_starts(members):
    """File offset of every member's gzip header (members are contiguous, the first at 0)."""
    ends = members[:, PAYLOAD_OFF] + members[:, PAYLOAD_LEN] + 8
    return np.r_[0, ends[:-1]].astype(np.int64)


def member_range(members, off, length):
    """Members [m0, m1) whose output covers text bytes [off, off + length)."""
    ends = members[:, OUT_OFF] + members[:, ISIZE]
    m0 = int(np.searchsorted(ends, off, side="right"))
    m1 = int(np.searchsorted(members[:, OUT_OFF], off + length, side="left"))
    return m0, max(m0, m1)


def sub_table(buf, members, m0, m1):
    """(compressed bytes, member table) of members [m0, m1) on their own: payload and output offsets rebased."""
    if m1 <= m0:
        return b"", np.zeros((0, 5), np.int64)
    lo = int(member_starts(members)[m0])
    hi = int(members[m1 - 1, PAYLOAD_OFF] + members[m1 - 1, PAYLOAD_LEN] + 8)
    sub = members[m0:m1].copy()
    sub[:, PAYLOAD_OFF] -= lo
    sub[:, OUT_OFF] -= sub[0, OUT_OFF]
    return bytes(buf[lo:hi]), sub


class BgzfReader:
    """Read-only, seekable view of a BGZF file's text.  Members are inflated on the host (zlib) only as reads reach
    them, so the chunk scanner can look around its cut points without inflating the file."""

    def __init__(self, buf, members):
        self._buf, self._m = buf, members
        self._ends = members[:, OUT_OFF] + members[:, ISIZE]
        self._starts = member_starts(members)
        self.size = text_size(members)
        self._pos = 0
        self._cache = {}

    def _member(self, i):
        data = self._cache.get(i)
        if data is None:   # the whole member through gzip: a bad one raises what reading the file with gzip raises
            hi = int(self._m[i, PAYLOAD_OFF] + self._m[i, PAYLOAD_LEN] + 8)
            data = gzip.decompress(bytes(self._buf[int(self._starts[i]):hi]))
            if len(self._cache) > 64:
                self._cache.clear()
            self._cache[i] = data
        return data

    def seek(self, pos):
        self._pos = pos

    def read(self, n):
        lo, hi = self._pos, min(self._pos + n, self.size)
        if lo >= hi:
            return b""
        parts = []
        i = int(np.searchsorted(self._ends, lo, side="right"))
        while lo < hi:
            base = int(self._m[i, OUT_OFF])
            data = self._member(i)
            take = data[lo - base:hi - base]
            parts.append(take)
            lo += len(take)
            i += 1
        self._pos = hi
        return b"".join(parts)
