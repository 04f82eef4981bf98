"""The Deflate64 parity reference itself: the Python decoder against zlib (DEFLATE mode), the C encoder's round trips, and
known-answer Deflate64 streams assembled bit by bit here, whose expected bytes are built directly (no decoder involved)."""
import random
import zlib

import pytest

from otezip_b200 import synth
from tests.deflate64 import inflate, Encoder


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

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)
        return self

    def done(self):
        return bytes(self.align().out)


def fixed_lit(w, s):
    if s < 144:
        return w.code(0x30 + s, 8)
    if s < 256:
        return w.code(0x190 + s - 144, 9)
    if s < 280:
        return w.code(s - 256, 7)
    return w.code(0xC0 + s - 280, 8)


def fixed_dist(w, s, xb=0, xv=0):
    w.code(s, 5)
    return w.bits(xv, xb) if xb else w


def stored(w, data, final=0):
    w.bits(final, 1).bits(0, 2).align()
    w.bits(len(data), 16).bits(~len(data) & 0xFFFF, 16)
    for b in data:
        w.bits(b, 8)
    return w


def canon(lens):
    cnt = [0] * 16
    for l in lens:
        cnt[l] += 1
    cnt[0] = 0
    nxt, c = [0] * 16, 0
    for l in range(1, 16):
        c = (c + cnt[l - 1]) << 1
        nxt[l] = c
    out = {}
    for s, l in enumerate(lens):
        if l:
            out[s] = (nxt[l], l)
            nxt[l] += 1
    return out


def known_answers():
    """-> [(name, stream, expected bytes)]"""
    ka = []
    # symbol 285 with extra 0 (length 3) and 0xFFFF (length 65,538), both at distance 1
    w = BitW().bits(1, 1).bits(1, 2)
    fixed_lit(w, ord("a"))
    fixed_lit(w, 285).bits(0, 16)
    fixed_dist(w, 0)
    fixed_lit(w, 256)
    ka.append(("len3", w.done(), b"a" * 4))
    w = BitW().bits(1, 1).bits(1, 2)
    fixed_lit(w, ord("b"))
    fixed_lit(w, 285).bits(0xFFFF, 16)
    fixed_dist(w, 0)
    fixed_lit(w, 256)
    ka.append(("len65538_dist1", w.done(), b"b" * 65539))
    # distance symbols 30 / 31 at their minimum and maximum, behind a stored block of 65,535 bytes + 1 literal
    pre = synth.random_bytes(65535, 9)
    w = stored(BitW(), pre).bits(1, 1).bits(1, 2)
    fixed_lit(w, 0x5A)
    exp = bytearray(pre + b"\x5a")
    for sym, xv, d in ((30, 0, 32769), (30, 16383, 49152), (31, 0, 49153), (31, 16383, 65536)):
        # 285 extra 7 = length 10; each distance counts from the current end
        fixed_lit(w, 285).bits(7, 16)
        fixed_dist(w, sym, 14, xv)
        for _ in range(10):
            exp.append(exp[-d])
    # a long copy at distance 65,536 (2,000 bytes: several 258-byte pieces, source in HBM)
    fixed_lit(w, 285).bits(1997, 16)
    fixed_dist(w, 31, 14, 16383)
    for _ in range(2000):
        exp.append(exp[-65536])
    fixed_lit(w, 256)
    ka.append(("dist30_31_stored", w.done(), bytes(exp)))
    # a dynamic block with HDIST = 32 (every distance code 5 bits long) and HLIT = 286
    lit = [8] * 255 + [0] + [9] + [0] * 28 + [9]         # 0..254: 8 bits, 256 / 285: 9 bits -> complete
    dst = [5] * 32
    pc = canon([2, 0, 0, 0, 0, 2, 0, 0, 2, 2] + [0] * 9)  # code-length code over {0, 5, 8, 9}
    lc, dc = canon(lit), canon(dst)
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5]
    pl = {0: 2, 5: 2, 8: 2, 9: 2}
    w = BitW().bits(1, 1).bits(2, 2).bits(286 - 257, 5).bits(32 - 1, 5).bits(len(order) - 4, 4)
    for s in order:
        w.bits(pl.get(s, 0), 3)
    for l in lit + dst:
        w.code(*pc[l])
    for ch in b"AB":
        w.code(*lc[ch])
    w.code(*lc[285]).bits(5, 16)          # length 8
    w.code(*dc[1])                        # distance 2
    w.code(*lc[ord("C")])
    w.code(*lc[285]).bits(3 - 3, 16)      # length 3
    w.code(*dc[31]).bits(0, 14)           # distance 49,153: before the start of the output -> error, so use it only last
    ka_dyn_bad = w.code(*lc[256]).done()
    w = BitW().bits(1, 1).bits(2, 2).bits(286 - 257, 5).bits(32 - 1, 5).bits(len(order) - 4, 4)
    for s in order:
        w.bits(pl.get(s, 0), 3)
    for l in lit + dst:
        w.code(*pc[l])
    for ch in b"AB":
        w.code(*lc[ch])
    w.code(*lc[285]).bits(5, 16)
    w.code(*dc[1])
    w.code(*lc[256])
    ka.append(("dynamic_hdist32", w.done(), b"AB" * 5))
    return ka, ka_dyn_bad


KA, KA_BAD = known_answers()


@pytest.mark.parametrize("i", range(len(KA)), ids=[k[0] for k in KA])
def test_known_answers(i):
    name, stream, exp = KA[i]
    got, v = inflate(stream, len(exp))
    assert v == "ok" and got == exp, name
    # the same stream as DEFLATE means something else or nothing
    got8, v8 = inflate(stream, len(exp), "deflate")
    assert (got8, v8) != (exp, "ok"), name


def test_known_answer_errors():
    assert inflate(KA_BAD, 100)[1] == "data"          # distance 49,153 with 13 bytes of output
    name, stream, exp = KA[1]
    assert inflate(stream, len(exp) - 1)[1] == "overflow"
    got, v = inflate(stream, len(exp) + 5)
    assert v == "short" and got == exp
    for cut in (1, 2, 3, len(stream) - 1):
        assert inflate(stream[:cut], len(exp))[1] in ("truncated", "data"), cut
    assert inflate(b"", 10) == (b"", "truncated")
    # fixed-table symbols 286 / 287 and a dynamic header with HLIT = 287
    for s in (286, 287):
        w = BitW().bits(1, 1).bits(1, 2)
        fixed_lit(w, s)
        assert inflate(w.done(), 10)[1] == "data"
    assert inflate(BitW().bits(1, 1).bits(2, 2).bits(30, 5).bits(0, 5).bits(0, 4).done() + bytes(8), 10)[1] == "data"


@pytest.mark.parametrize("strategy", [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED])
def test_deflate_mode_equals_zlib(strategy):
    rnd = random.Random(strategy)
    for k in range(6):
        data = synth.jsonlog_text(rnd.randint(0, 200000), k) + synth.random_bytes(rnd.randint(0, 3000), k) + b"z" * rnd.randint(0, 70000)
        c = zlib.compressobj(rnd.choice([0, 1, 6, 9]), zlib.DEFLATED, -15, 8, strategy)
        z = c.compress(data) + c.flush()
        assert inflate(z, len(data), "deflate") == (zlib.decompress(z, -15), "ok")


@pytest.mark.parametrize("mode", ["deflate64", "dual", "deflate"])
@pytest.mark.parametrize("block", ["dynamic", "fixed", "stored", "mixed"])
def test_encoder_round_trip(mode, block):
    E = Encoder()
    blob = synth.random_bytes(40000, 3)
    for data in (b"", b"q", synth.jsonlog_text(150000, 1), synth.random_bytes(70000, 2), b"x" * 140000, blob * 4 + blob[:999]):
        c = E.compress(data, mode, block)
        if mode != "deflate64":
            assert zlib.decompress(c, -15) == data
        for m in (("deflate64", "deflate") if mode == "dual" else ("deflate" if mode == "deflate" else "deflate64",)):
            assert inflate(c, len(data), m) == (data, "ok"), (m, len(data))


def test_encoder_writes_what_only_deflate64_has():
    """64 KiB window and long matches: zlib must reject the stream (or decode something else)"""
    blob = synth.random_bytes(50000, 7)
    data = blob + b"-" + blob + b"r" * 100000
    c = Encoder().compress(data, "deflate64")
    assert inflate(c, len(data)) == (data, "ok")
    try:
        assert zlib.decompress(c, -15) != data
    except zlib.error:
        pass
