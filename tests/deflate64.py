"""Plain-Python Deflate64 / DEFLATE decoder: the parity reference for ZIP method 9, which the reference library rejects.

inflate(data, cap, mode) decodes one raw stream into at most `cap` bytes and returns (bytes, verdict), verdict one of
"ok", "short" (valid stream that ends before `cap` bytes), "data", "truncated", "overflow" — the classes of the status
words OTZ_ST_OK, OTZ_ST_OK | OTZ_STF_SHORT, OTZ_ST_DATA, OTZ_ST_TRUNCATED, OTZ_ST_OVERFLOW.  The bytes are what was
produced up to the verdict.  The decoder is strict in the same places as k_inflate: incomplete code sets are rejected
except a single 1-bit code, HLIT > 286 and (DEFLATE) HDIST > 30 are errors, a distance may not reach before the start of
the output.  Bits past the end of the input read as zero, and the end of the input is tested after every header, table
and symbol, as the kernel tests it.

mode="deflate64" (PKWARE's enhanced deflate; zlib contrib/infback9): 64 KiB window, length symbol 285 = 3 + 16 extra bits,
distance symbols 30 / 31 = 32,769 / 49,153 + 14 extra bits, HDIST up to 32.  mode="deflate": RFC 1951.

Encoder: the C encoder of tools/d64enc.c (hash-chain LZ77, fixed / dynamic / stored blocks), loaded by ctypes."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENC_SO = os.path.join(ROOT, "tools", "libd64enc.so")

_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227]
_LEN_XB = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5]
_DST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577, 32769, 49153]
_DST_XB = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13, 14, 14]
_CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


class _Err(Exception):
    def __init__(self, verdict):
        self.verdict = verdict


class _Bits:
    def __init__(self, data: bytes):
        self.d = data
        self.total = 8 * len(data)
        self.pos = 0

    def get(self, n: int) -> int:
        p = self.pos
        i = p >> 3
        chunk = int.from_bytes(self.d[i:i + 8], "little")   # (past the end: zero bits)
        self.pos = p + n
        return (chunk >> (p & 7)) & ((1 << n) - 1)

    def peek(self, n: int) -> int:
        p = self.pos
        i = p >> 3
        return (int.from_bytes(self.d[i:i + 4], "little") >> (p & 7)) & ((1 << n) - 1)

    def rem(self) -> int:
        return self.total - self.pos


def _table(lens, allow_empty: bool):
    """-> (lookup list indexed by the next `maxlen` stream bits -> (symbol, length) or None, maxlen); None = invalid set"""
    cnt = [0] * 16
    for l in lens:
        cnt[l] += 1
    cnt[0] = 0
    left, ncodes = 1, 0
    for l in range(1, 16):
        left = (left << 1) - cnt[l]
        if left < 0:
            return None
        ncodes += cnt[l]
    if ncodes == 0:
        return ([None], 0) if allow_empty else None
    if left > 0 and not (ncodes == 1 and cnt[1] == 1):
        return None
    maxlen = max(l for l in lens if l)
    nxt, code = [0] * 16, 0
    for l in range(1, 16):
        code = (code + cnt[l - 1]) << 1 if l > 1 else 0
        nxt[l] = code
    tab = [None] * (1 << maxlen)
    for s, l in enumerate(lens):
        if not l:
            continue
        c = nxt[l]
        nxt[l] += 1
        rev = int(format(c, "0%db" % l)[::-1], 2)
        for k in range(rev, 1 << maxlen, 1 << l):
            tab[k] = (s, l)
    return tab, maxlen


def _decode(br: _Bits, t) -> int:
    tab, maxlen = t
    e = tab[br.peek(maxlen)] if maxlen else None
    if e is None:
        raise _Err("data")
    br.pos += e[1]
    return e[0]


_FIXED = (_table([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8, False), _table([5] * 32, True))


def _dynamic(br: _Bits, d64: bool):
    hlit, hdist, hclen = br.get(5) + 257, br.get(5) + 1, br.get(4) + 4
    if hlit > 286 or (not d64 and hdist > 30):
        raise _Err("data")
    cl = [0] * 19
    for i in range(hclen):
        cl[_CL_ORDER[i]] = br.get(3)
    cnt = [0] * 8
    for l in cl:
        cnt[l] += 1
    left = 1
    for l in range(1, 8):
        left = (left << 1) - cnt[l]
        if left < 0:
            raise _Err("data")
    if left != 0:
        raise _Err("data")          # the code-length code must be complete
    pre = _table(cl, False)
    lens, prev, total = [], 0, hlit + hdist
    while len(lens) < total:
        sym = _decode(br, pre)
        if sym < 16:
            lens.append(sym)
            prev = sym
            continue
        if sym == 16:
            if not lens:
                raise _Err("data")
            val, rep = prev, 3 + br.get(2)
        elif sym == 17:
            val, rep = 0, 3 + br.get(3)
        else:
            val, rep = 0, 11 + br.get(7)
        if len(lens) + rep > total:
            raise _Err("data")
        lens += [val] * rep
        prev = val
    if lens[256] == 0:
        raise _Err("data")
    lt = _table(lens[:hlit], False)
    if lt is None:
        raise _Err("data")
    dt = _table(lens[hlit:], True)
    if dt is None:
        raise _Err("data")
    return lt, dt


def inflate(data: bytes, cap: int, mode: str = "deflate64"):
    assert mode in ("deflate64", "deflate")
    d64 = mode == "deflate64"
    out = bytearray()
    if len(data) == 0:
        return b"", "truncated"
    br = _Bits(bytes(data))
    try:
        while True:
            final, btype = br.get(1), br.get(2)
            if br.rem() < 0:
                raise _Err("truncated")
            if btype == 0:
                pos = (br.pos + 7) >> 3
                if len(data) - pos < 4:
                    raise _Err("data")
                ln = data[pos] | data[pos + 1] << 8
                nln = data[pos + 2] | data[pos + 3] << 8
                if ln != (~nln & 0xFFFF) or len(data) - pos - 4 < ln:
                    raise _Err("data")
                if cap - len(out) < ln:
                    raise _Err("overflow")
                out += data[pos + 4:pos + 4 + ln]
                br.pos = 8 * (pos + 4 + ln)
                if final:
                    break
                continue
            if btype == 3:
                raise _Err("data")
            if btype == 1:
                lt, dt = _FIXED   # (literal 286 / 287 and, in DEFLATE, distance 30 / 31 are rejected when decoded)
            else:
                lt, dt = _dynamic(br, d64)
            if br.rem() < 0:
                raise _Err("truncated")
            while True:
                sym = _decode(br, lt)
                if sym < 256:
                    if len(out) >= cap:
                        raise _Err("overflow")
                    out.append(sym)
                elif sym == 256:
                    break
                else:
                    v = sym - 257
                    if v >= 29:
                        raise _Err("data")
                    if v == 28:
                        length = 3 + br.get(16) if d64 else 258
                    else:
                        length = _LEN_BASE[v] + br.get(_LEN_XB[v])
                    ds = _decode(br, dt)
                    if ds >= (32 if d64 else 30):
                        raise _Err("data")
                    dist = _DST_BASE[ds] + br.get(_DST_XB[ds])
                    if dist > len(out):
                        raise _Err("data")
                    if length > cap - len(out):
                        raise _Err("overflow")
                    if dist >= length:
                        s = len(out) - dist
                        out += out[s:s + length]
                    else:
                        pat = bytes(out[len(out) - dist:])
                        out += (pat * (length // dist + 1))[:length]
                if br.rem() < 0:
                    raise _Err("truncated")
            if br.rem() < 0:
                raise _Err("truncated")
            if final:
                break
    except _Err as e:
        return bytes(out), e.verdict
    return bytes(out), "ok" if len(out) == cap else "short"


# ---------------------------------------------------------------- the C encoder
MODES = {"deflate64": 0, "dual": 1, "deflate": 2}
BLOCKS = {"dynamic": 0, "fixed": 1, "stored": 2, "mixed": 3}


def build_encoder() -> None:
    subprocess.run(["make", "-C", ROOT, "tools/libd64enc.so"], check=True, stdout=subprocess.DEVNULL)


class Encoder:
    """deflate64: 64 KiB window, matches up to 65,538 bytes.  dual: 32 KiB window, matches up to 257 bytes — a stream that
    decodes to the same bytes as Deflate64 and as DEFLATE (only length 258, symbol 285, is coded differently).  deflate:
    RFC 1951.  chain = hash-chain candidates per position; block = dynamic / fixed / stored / mixed (cycles the three)."""

    def __init__(self):
        if not os.path.exists(ENC_SO):
            build_encoder()
        self.L = C.CDLL(ENC_SO)
        self.L.d64enc.restype = C.c_int64
        self.L.d64enc.argtypes = [C.c_char_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int]
        self.L.d64enc_bound.restype = C.c_uint64
        self.L.d64enc_bound.argtypes = [C.c_uint64]

    def compress(self, data: bytes, mode: str = "deflate64", block: str = "dynamic", chain: int = 32) -> bytes:
        cap = self.L.d64enc_bound(len(data))
        buf = C.create_string_buffer(cap)
        n = self.L.d64enc(data, len(data), buf, cap, MODES[mode], BLOCKS[block], chain)
        if n < 0:
            raise RuntimeError("d64enc failed (%d)" % n)
        return buf.raw[:n]
