"""LZ77 records on the edges of k_inflate_lz's match descriptor, in hand-assembled fixed-Huffman DEFLATE streams.

The executor runs a match on its common path (two loads and two stores per lane) only when it is at most 64 elements
long, does not overlap itself, neither range wraps around the ring and its source does not reach into what the same
batch writes; everything else takes a side path.  The streams below put records on every one of those edges: lengths
3 / 31 / 32 / 33 / 63 / 64 / 65 / 258; distances 1, len - 1, len, len + 1; sources that end exactly at, or one element
past, the previous record's destination; sources just inside and just outside the ring (4 / 8 / 16 KiB) and far ones;
long literal runs and runs of far matches that end batches at the output span and at the staging budget.  Each pattern
runs in a small entry (byte executor) and repeated into an entry of more than 2 MiB (segmented execution over 16-bit
symbols), against zlib and the oracle, and once more against the bounds-checked build with every counter at zero."""
import json
import os
import random
import subprocess
import sys
import zlib

import numpy as np
import pytest

from otezip_b200 import Ctx, synth
from otezip_b200.native import parse_central, default_opts

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DBG = os.path.join(ROOT, "otezip_b200", "libotezip_b200_dbg.so")

_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
_LEN_XB = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
_DST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
             8193, 12289, 16385, 24577]
_DST_XB = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]


class BitW:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v, n):            # LSB first (header fields, extra bits)
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8
        return self

    def code(self, c, n):            # Huffman code, most significant bit first
        return self.bits(int(format(c, "0%db" % n)[::-1], 2), n)

    def done(self):
        if self.n:
            self.bits(0, 8 - self.n)
        return bytes(self.out)


def _lit(w, s):
    if s < 144:
        return w.code(0x30 + s, 8)
    if s < 256:
        return w.code(0x190 + s - 144, 9)
    if s < 280:
        return w.code(s - 256, 7)
    return w.code(0xC0 + s - 280, 8)


def _sym(base, v):
    i = max(k for k, b in enumerate(base) if b <= v)
    return i, v - base[i]


def encode(tokens, block=20000):
    """fixed-Huffman blocks from a token list: an int is a literal byte, (length, distance) a match.  The final block is
    an empty stored block, a tail the reference's inflater always accepts (SURVEY.md F1), so the oracle checks every
    stream."""
    w = BitW()
    for b0 in range(0, max(len(tokens), 1), block):
        part = tokens[b0:b0 + block]
        w.bits(0, 1).bits(1, 2)
        for t in part:
            if isinstance(t, int):
                _lit(w, t)
                continue
            ln, d = t
            i, x = _sym(_LEN_BASE, ln) if ln != 258 else (28, 0)
            _lit(w, 257 + i)
            if _LEN_XB[i]:
                w.bits(x, _LEN_XB[i])
            j, y = _sym(_DST_BASE, d)
            w.code(j, 5)
            if _DST_XB[j]:
                w.bits(y, _DST_XB[j])
        _lit(w, 256)
    w.bits(1, 1).bits(0, 2).done()           # BFINAL stored block of length 0
    w.bits(0, 16).bits(0xFFFF, 16)
    return w.done()


def expand(tokens):
    out = bytearray()
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        else:
            ln, d = t
            for _ in range(ln):
                out.append(out[-d])
    return bytes(out)


LENGTHS = [3, 31, 32, 33, 63, 64, 65, 258]
RINGS = [4096, 8192, 16384]


def records(seed, n_out):
    """a seeded record mix that keeps hitting the edges listed above until n_out bytes are out"""
    rnd = random.Random(seed)
    toks = [rnd.randrange(256) for _ in range(40000)]   # history for every far distance
    pos, prev = len(toks), (len(toks) - 1, 1)           # prev: (destination, length) of the previous match
    while pos < n_out:
        kind = rnd.randrange(9)
        if kind == 0:                                   # literal runs that end batches at the output span
            run = rnd.choice([0, 1, 4, 5, 200, 511, 512, 700, 1100])
        else:
            run = rnd.choice([0, 0, 0, 1, 2, 3])
        toks += [rnd.randrange(256) for _ in range(run)]
        pos += run
        if kind == 1:                                   # a burst of long far matches: the staging budget ends the batch
            for _ in range(rnd.randint(3, 12)):
                ln = rnd.choice([64, 65, 200, 258])
                d = rnd.choice([20000, 30000, 32768])
                toks.append((ln, d))
                prev = (pos, ln)
                pos += ln
            continue
        ln = rnd.choice(LENGTHS)
        if kind in (2, 3):                              # overlap edges: periodic or not
            d = rnd.choice([1, max(ln - 1, 1), ln, ln + 1])
        elif kind == 4:                                 # the source ends at / one element past the previous destination
            end = prev[0] + prev[1] + rnd.choice([-1, 0, 1])
            d = max(pos - (end - ln), 1)
        elif kind == 5:                                 # just inside / just outside each ring size
            w = rnd.choice(RINGS)
            d = w + rnd.choice([-1300, -1024, -700, -ln - 1, -ln, -1, 0, 1, 600, 1100])
        elif kind == 6:                                 # far
            d = rnd.choice([4097, 8193, 16385, 24577, 32768])
        else:                                           # near, often wrapping the ring on one side or both
            d = rnd.choice([ln + 2, 100, 700, 1000, 2000, 3000])
        d = max(1, min(d, pos, 32768))
        toks.append((ln, d))
        prev = (pos, ln)
        pos += ln
    return toks


def _member(name, toks):
    raw = expand(toks)
    payload = encode(toks)
    assert zlib.decompress(payload, -15) == raw
    return synth.Member(name, 8, payload, len(raw), zlib.crc32(raw) & 0xFFFFFFFF, raw=raw)


def _archive():
    ms = []
    for s in range(4):
        ms.append(_member("small%d" % s, records(10 + s, 150000)))      # byte executor
    for s in range(2):
        ms.append(_member("huge%d" % s, records(20 + s, 2600000)))      # segmented, over 16-bit symbols
    return ms


def _extract(ms, env=None):
    img = synth.build_zip(ms)
    tab = parse_central(img)
    os.environ.update(env or {})
    try:
        c = Ctx(0)
        out, crc, st = c.extract_host(img, tab, default_opts())
        fb = int(c.L.otz_inflate_fallbacks(c.h))
        c.close()
    finally:
        for k in env or {}:
            del os.environ[k]
    return img, tab, out, crc, st, fb


@pytest.mark.parametrize("ring", [None, "8192", "16384"])
def test_edge_records_match_zlib_and_oracle(ring):
    from oracle import Oracle
    ms = _archive()
    img, tab, out, crc, st, fb = _extract(ms, {"OTZ_LZ_RING": ring} if ring else {})
    assert fb == 0, fb   # every stream went through the two-phase path
    o = Oracle()
    rc, oents = o.load_central(img)
    ost, ocrc, oout, oofs = o.extract_all(img, oents)
    for i, m in enumerate(ms):
        assert int(st[i]) == 0 and ost[i] == 0, (m.name, hex(int(st[i])), int(ost[i]))
        a = out[int(tab["out_ofs"][i]):int(tab["out_ofs"][i]) + m.uncomp_size]
        assert np.array_equal(a, np.frombuffer(m.raw, np.uint8)), (m.name, int(np.argmax(a != np.frombuffer(m.raw, np.uint8))))
        assert np.array_equal(a, oout[int(oofs[i]):int(oofs[i]) + m.uncomp_size]), m.name
        assert int(crc[i]) == int(ocrc[i]) == m.crc32, m.name


CHILD = r'''
import ctypes as C, json, sys
sys.path.insert(0, %(root)r)
import numpy as np
from otezip_b200.native import Lib
from tests.test_gpu_lz_records import _archive, _extract
L = Lib.get().L
L.otz_debug_violations.argtypes = [C.c_void_p, C.c_int]
ms = _archive()
bad = 0
for env in ({}, {"OTZ_LZ_RING": "16384", "OTZ_SEG_PAR_RING": "8192"}):
    img, tab, out, crc, st, fb = _extract(ms, env)
    for i, m in enumerate(ms):
        a = out[int(tab["out_ofs"][i]):int(tab["out_ofs"][i]) + m.uncomp_size]
        bad += int(st[i]) != 0 or not np.array_equal(a, np.frombuffer(m.raw, np.uint8))
v = (C.c_uint64 * 32)()
n = L.otz_debug_violations(v, 32)
print(json.dumps({"slots": n, "violations": [int(x) for x in v[:max(n, 0)]], "mismatches": bad}))
'''


@pytest.mark.skipif(not os.path.exists(DBG), reason="debug library not built (make debug)")
def test_edge_records_bounds_checked_build():
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, OTEZIP_B200_LIB=DBG))
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["slots"] > 0 and d["mismatches"] == 0 and sum(d["violations"]) == 0, d
