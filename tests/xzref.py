"""Plain-Python xz / LZMA2 / LZMA decoder: the parity reference for ZIP method 95 (XZ), which the reference library rejects.

decode(payload, cap) decodes a method-95 payload (one or more xz streams, with stream padding) into at most `cap` bytes and
returns (bytes, verdict), verdict one of "ok", "short" (valid payload that ends before `cap` bytes), "data", "truncated",
"overflow", "method" -- the classes of OTZ_ST_OK, OTZ_ST_OK | OTZ_STF_SHORT, OTZ_ST_DATA, OTZ_ST_TRUNCATED,
OTZ_ST_OVERFLOW, OTZ_ST_METHOD.  The bytes are what was produced before the verdict.

It is written as k_xz.cuh is built: walk() parses the container and hops the LZMA2 chunk headers without decoding them,
validating everything structural and stopping at the first structural error; the chunks it accepted are then decoded in
order, and an error inside a chunk wins over the walk's error, which comes later in the stream.  The check field of a block
(CRC32 / CRC64 / SHA-256) is skipped, not verified: the ZIP CRC-32 covers the entry.

What is verified: the CRC32 of the stream header, of every block header, of the index and of the footer; the index against
the blocks (record count, unpadded and unpacked sizes); the footer's backward size against the index; the sizes a block
header carries against its block; stream padding (zero bytes, a multiple of 4).  What is rejected as "method": a filter
chain other than exactly one LZMA2 filter.  The LZMA2 rules are liblzma's: the first chunk of a block resets the dictionary,
lc + lp <= 4 and pb <= 4, the first LZMA chunk after a dictionary reset carries properties, an LZMA chunk ends with its range
coder exactly at its packed size with code == 0, no end-of-stream marker, and a match distance is below
min(dict_size, bytes produced since the last dictionary reset)."""
from __future__ import annotations

import zlib

MAGIC = b"\xfd7zXZ\x00"
FOOTER_MAGIC = b"YZ"
CHECK_SIZE = {0: 0, 1: 4, 4: 8, 10: 32}   # check IDs None, CRC32, CRC64, SHA-256; the others are reserved
FILTER_LZMA2 = 0x21


class _Err(Exception):
    def __init__(self, verdict):
        self.verdict = verdict


def dict_size(code: int) -> int:
    """LZMA2 filter property byte (code <= 40) -> dictionary size"""
    return 0xFFFFFFFF if code == 40 else (2 | (code & 1)) << (code // 2 + 11)


class _In:
    def __init__(self, d: bytes):
        self.d = d
        self.p = 0

    def need(self, n: int):
        if self.p + n > len(self.d):
            raise _Err("truncated")

    def byte(self) -> int:
        self.need(1)
        self.p += 1
        return self.d[self.p - 1]

    def take(self, n: int) -> bytes:
        self.need(n)
        self.p += n
        return self.d[self.p - n:self.p]

    def vli(self) -> int:
        v = 0
        for i in range(9):
            b = self.byte()
            v |= (b & 0x7F) << (7 * i)
            if not b & 0x80:
                if b == 0 and i > 0:
                    raise _Err("data")   # not the shortest encoding
                return v
        raise _Err("data")


def walk(payload: bytes, cap: int):
    """-> (chunks, verdict).  chunks: (kind, data offset, packed, unpacked, props or None, reset, dict_size) in stream order,
    kind "lzma" or "copy", reset = "dict" / "state" / None, props = (lc, lp, pb) of a chunk that sets them.  verdict: "ok" or the first structural
    error; the chunks are those before it."""
    chunks = []
    r = _In(payload)
    out = 0
    try:
        if not payload:
            raise _Err("truncated")
        while True:
            # ---- stream header
            hdr = r.take(12)
            if hdr[:6] != MAGIC or zlib.crc32(hdr[6:8]) != int.from_bytes(hdr[8:12], "little"):
                raise _Err("data")
            flags = hdr[6:8]
            if flags[0] != 0 or flags[1] & 0xF0 or (flags[1] & 15) not in CHECK_SIZE:
                raise _Err("data")
            csize = CHECK_SIZE[flags[1] & 15]
            records = []
            while True:
                b0 = r.byte()
                if b0 == 0:
                    break   # index indicator
                # ---- block header
                hstart = r.p - 1
                hsize = (b0 + 1) * 4
                r.need(hsize - 1)
                h = payload[hstart:hstart + hsize]
                if zlib.crc32(h[:-4]) != int.from_bytes(h[-4:], "little"):
                    raise _Err("data")
                bf = r.byte()
                if bf & 0x3C:
                    raise _Err("data")
                nfilt = (bf & 3) + 1
                hcomp = r.vli() if bf & 0x40 else None
                hunc = r.vli() if bf & 0x80 else None
                fid = r.vli()
                npr = r.vli()
                if r.p + npr > hstart + hsize - 4:
                    raise _Err("data")
                prop = r.take(npr)
                if nfilt != 1 or fid != FILTER_LZMA2:
                    raise _Err("method")
                if npr != 1 or prop[0] > 40:
                    raise _Err("data")
                if r.p > hstart + hsize - 4 or any(payload[r.p:hstart + hsize - 4]) or hcomp == 0:
                    raise _Err("data")
                dsz = dict_size(prop[0])
                r.p = hstart + hsize
                # ---- LZMA2 chunks
                dstart = r.p
                bunc = 0
                need_dict, need_props = True, True
                props = None
                while True:
                    c = r.byte()
                    if c == 0:
                        break
                    if c == 1 or c >= 0xE0:
                        need_dict, need_props = False, True
                        reset = "dict"
                    elif need_dict:
                        raise _Err("data")
                    else:
                        reset = None
                    if c >= 0x80:
                        unp = ((c & 0x1F) << 16) + (r.byte() << 8) + r.byte() + 1
                        pk = (r.byte() << 8) + r.byte() + 1
                        if c >= 0xC0:
                            p = r.byte()
                            if p > 224:
                                raise _Err("data")
                            lc, lp, pb = p % 9, p // 9 % 5, p // 45
                            if lc + lp > 4:
                                raise _Err("data")
                            props = (lc, lp, pb)
                            need_props = False
                        elif need_props:
                            raise _Err("data")
                        if reset is None and c >= 0xA0:
                            reset = "state"
                        if out + unp > cap:
                            raise _Err("overflow")
                        r.need(pk)
                        chunks.append(("lzma", r.p, pk, unp, props if c >= 0xC0 else None, reset, dsz))
                        r.p += pk
                    elif c <= 2:
                        unp = (r.byte() << 8) + r.byte() + 1
                        if out + unp > cap:
                            raise _Err("overflow")
                        r.need(unp)
                        chunks.append(("copy", r.p, unp, unp, None, reset, dsz))
                        r.p += unp
                    else:
                        raise _Err("data")
                    out += unp
                    bunc += unp
                bcomp = r.p - dstart
                if (hcomp is not None and hcomp != bcomp) or (hunc is not None and hunc != bunc):
                    raise _Err("data")
                if any(r.take((-(r.p - hstart)) % 4)):
                    raise _Err("data")
                r.take(csize)
                records.append((hsize + bcomp + csize, bunc))
            # ---- index
            istart = r.p - 1
            if r.vli() != len(records):
                raise _Err("data")
            for unpadded, unc in records:
                if r.vli() != unpadded or r.vli() != unc:
                    raise _Err("data")
            if any(r.take((-(r.p - istart)) % 4)):
                raise _Err("data")
            crc = r.take(4)
            if zlib.crc32(payload[istart:r.p - 4]) != int.from_bytes(crc, "little"):
                raise _Err("data")
            # ---- footer
            f = r.take(12)
            if zlib.crc32(f[4:10]) != int.from_bytes(f[:4], "little") or f[10:12] != FOOTER_MAGIC or f[8:10] != flags:
                raise _Err("data")
            if (int.from_bytes(f[4:8], "little") + 1) * 4 != r.p - 12 - istart:
                raise _Err("data")
            # ---- stream padding (zero bytes, a multiple of 4), then the end or another stream
            z = r.p
            while r.p < len(payload) and payload[r.p] == 0:
                r.p += 1
            if (r.p - z) % 4:
                raise _Err("data")
            if r.p == len(payload):
                return chunks, "ok"
    except _Err as e:
        return chunks, e.verdict


class _Rc:
    def __init__(self, d: bytes, lo: int, hi: int):
        if hi - lo < 5 or d[lo] != 0:
            raise _Err("data")
        self.d, self.p, self.hi = d, lo + 5, hi
        self.code = int.from_bytes(d[lo + 1:lo + 5], "big")
        self.range = 0xFFFFFFFF

    def norm(self):
        if self.range < (1 << 24):
            if self.p >= self.hi:
                raise _Err("data")   # the chunk's packed size is used up
            self.range = (self.range << 8) & 0xFFFFFFFF
            self.code = ((self.code << 8) | self.d[self.p]) & 0xFFFFFFFF
            self.p += 1

    def bit(self, probs, i) -> int:
        self.norm()
        p = probs[i]
        bound = (self.range >> 11) * p
        if self.code < bound:
            self.range = bound
            probs[i] = p + ((2048 - p) >> 5)
            return 0
        self.range -= bound
        self.code -= bound
        probs[i] = p - (p >> 5)
        return 1

    def direct(self, n: int) -> int:
        v = 0
        for _ in range(n):
            self.norm()
            self.range >>= 1
            b = 1 if self.code >= self.range else 0
            if b:
                self.code -= self.range
            v = (v << 1) | b
        return v

    def tree(self, probs, base, nbits) -> int:
        m = 1
        for _ in range(nbits):
            m = (m << 1) | self.bit(probs, base + m)
        return m - (1 << nbits)

    def rtree(self, probs, base, nbits) -> int:
        m, v = 1, 0
        for i in range(nbits):
            b = self.bit(probs, base + m)
            m = (m << 1) | b
            v |= b << i
        return v


# probability array layout (the kernel's too)
P_ISMATCH = 0                  # [state 12][pos_state 16]
P_ISREP = 192                  # [12]
P_ISREP0 = 204
P_ISREP1 = 216
P_ISREP2 = 228
P_ISREP0L = 240                # [12][16]
P_SLOT = 432                   # [len_state 4][64]
P_SPEC = 688                   # 114 + 1 (index base dist - slot - 1 + m)
P_ALIGN = 803                  # [16]
P_LEN = 819                    # choice, choice2, low[16][8], mid[16][8], high[256]  = 514
P_REPLEN = 1333
P_LIT = 1847                   # [0x300 << (lc + lp)]
LEN_LOW, LEN_MID, LEN_HIGH = 2, 130, 258


class _Lzma:
    def __init__(self):
        self.probs = None

    def reset_state(self, lc, lp, pb):
        self.lc, self.lp, self.pb = lc, lp, pb
        self.probs = [1024] * (P_LIT + (0x300 << (lc + lp)))
        self.state = 0
        self.rep = [0, 0, 0, 0]

    def length(self, rc, base, ps) -> int:
        P = self.probs
        if not rc.bit(P, base):
            return 2 + rc.tree(P, base + LEN_LOW + ps * 8 - 1, 3)
        if not rc.bit(P, base + 1):
            return 10 + rc.tree(P, base + LEN_MID + ps * 8 - 1, 3)
        return 18 + rc.tree(P, base + LEN_HIGH - 1, 8)

    def chunk(self, out: bytearray, base: int, dsz: int, d: bytes, lo: int, pk: int, unp: int):
        """decode one LZMA chunk of `unp` bytes from d[lo, lo + pk) onto out; positions count from `base` (the last reset)"""
        rc = _Rc(d, lo, lo + pk)
        P = self.probs
        lc, lpm, pbm = self.lc, (1 << self.lp) - 1, (1 << self.pb) - 1
        end = len(out) + unp
        st, rep = self.state, self.rep
        while len(out) < end:
            pos = len(out) - base
            ps = pos & pbm
            if not rc.bit(P, P_ISMATCH + st * 16 + ps):
                prev = out[-1] if pos else 0
                li = P_LIT + 0x300 * (((pos & lpm) << lc) + (prev >> (8 - lc)))
                m = 1
                if st >= 7:
                    mb = out[len(out) - rep[0] - 1]
                    while m < 0x100:
                        mbit = (mb >> 7) & 1
                        mb <<= 1
                        b = rc.bit(P, li + 0x100 + (mbit << 8) + m)
                        m = (m << 1) | b
                        if b != mbit:
                            break
                while m < 0x100:
                    m = (m << 1) | rc.bit(P, li + m)
                out.append(m & 0xFF)
                st = 0 if st < 4 else st - 3 if st < 10 else st - 6
                continue
            if not rc.bit(P, P_ISREP + st):
                n = self.length(rc, P_LEN, ps)
                ls = min(n - 2, 3)
                slot = rc.tree(P, P_SLOT + ls * 64 - 1, 6)
                if slot < 4:
                    dist = slot
                else:
                    nd = (slot >> 1) - 1
                    dist = (2 | (slot & 1)) << nd
                    if slot < 14:
                        dist += rc.rtree(P, P_SPEC + dist - slot - 1, nd)
                    else:
                        dist += rc.direct(nd - 4) << 4
                        dist += rc.rtree(P, P_ALIGN - 1, 4)
                        if dist == 0xFFFFFFFF:
                            raise _Err("data")   # end-of-stream marker: not allowed in LZMA2
                rep[3], rep[2], rep[1], rep[0] = rep[2], rep[1], rep[0], dist
                st = 7 if st < 7 else 10
            else:
                if not rc.bit(P, P_ISREP0 + st):
                    if not rc.bit(P, P_ISREP0L + st * 16 + ps):
                        st = 9 if st < 7 else 11
                        n = 1
                        if rep[0] >= pos or rep[0] >= dsz:
                            raise _Err("data")
                        out.append(out[len(out) - rep[0] - 1])
                        continue
                else:
                    if not rc.bit(P, P_ISREP1 + st):
                        dist = rep[1]
                    else:
                        if not rc.bit(P, P_ISREP2 + st):
                            dist = rep[2]
                        else:
                            dist = rep[3]
                            rep[3] = rep[2]
                        rep[2] = rep[1]
                    rep[1] = rep[0]
                    rep[0] = dist
                n = self.length(rc, P_REPLEN, ps)
                st = 8 if st < 7 else 11
            if rep[0] >= pos or rep[0] >= dsz:
                raise _Err("data")
            if len(out) + n > end:
                raise _Err("data")   # a match across the end of the chunk
            s = len(out) - rep[0] - 1
            for i in range(n):
                out.append(out[s + i])
        self.state = st
        rc.norm()
        if rc.p != lo + pk or rc.code != 0:
            raise _Err("data")


def decode(payload: bytes, cap: int):
    """-> (bytes, verdict); see the module docstring"""
    chunks, verdict = walk(payload, cap)
    out = bytearray()
    lz = _Lzma()
    base = 0
    try:
        for kind, lo, pk, unp, props, reset, dsz in chunks:
            if reset == "dict":
                base = len(out)
            if props is not None:
                lz.reset_state(*props)
            elif reset == "state":
                lz.reset_state(lz.lc, lz.lp, lz.pb)
            if kind == "copy":
                out += payload[lo:lo + unp]
            else:
                lz.chunk(out, base, dsz, payload, lo, pk, unp)
    except _Err as e:
        return bytes(out), e.verdict
    if verdict != "ok":
        return bytes(out), verdict
    return bytes(out), "ok" if len(out) == cap else "short"
