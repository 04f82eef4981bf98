"""tests/xzref.py against liblzma (Python's lzma module, and `xz -t` where the case needs concatenated streams, padding or the
exact liblzma verdict), on valid and invalid method-95 payloads.  No GPU.

The case lists (valid_cases / invalid_cases) are shared with tests/test_gpu_xz.py."""
import hashlib
import lzma
import random
import shutil
import struct
import subprocess
import zlib

import pytest

from otezip_b200 import synth
from tests import xzref

XZ = shutil.which("xz")
CHECK_BYTES = {0: 0, 1: 4, 4: 8, 10: 32}


# ---------------------------------------------------------------------------------------------------- xz container builder
def vli(v: int) -> bytes:
    out = bytearray()
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    out.append(v)
    return bytes(out)


def raw_lzma2(data: bytes, **opt) -> bytes:
    """raw LZMA2 data (chunks + end byte 0x00) from liblzma"""
    f = {"id": lzma.FILTER_LZMA2, "preset": opt.pop("preset", 6)}
    f.update(opt)
    return lzma.compress(data, format=lzma.FORMAT_RAW, filters=[f])


def check_field(check: int, data: bytes) -> bytes:
    if check == 1:
        return struct.pack("<I", zlib.crc32(data))
    if check == 4:
        return struct.pack("<Q", lzma_crc64(data))
    if check == 10:
        return hashlib.sha256(data).digest()
    return b""


def lzma_crc64(data: bytes) -> int:
    poly, crc = 0xC96C5795D7870F42, 0xFFFFFFFFFFFFFFFF
    for b in data:
        crc ^= b
        for _ in range(8):
            crc = (crc >> 1) ^ (poly if crc & 1 else 0)
    return crc ^ 0xFFFFFFFFFFFFFFFF


def block_header(dict_code=22, comp=None, unc=None, filters=None, pad_extra=0) -> bytes:
    """filters: list of (id, props) (default: one LZMA2 filter with dict_code)"""
    filters = filters if filters is not None else [(0x21, bytes([dict_code]))]
    flags = (len(filters) - 1) | (0x40 if comp is not None else 0) | (0x80 if unc is not None else 0)
    body = bytes([flags]) + (vli(comp) if comp is not None else b"") + (vli(unc) if unc is not None else b"")
    for fid, pr in filters:
        body += vli(fid) + vli(len(pr)) + pr
    size = (1 + len(body) + 4 + 3) // 4 * 4 + 4 * pad_extra
    h = bytes([size // 4 - 1]) + body
    h += bytes(size - 4 - len(h))
    return h + struct.pack("<I", zlib.crc32(h))


def stream(blocks, check=1, index=None, flags=None):
    """blocks: list of (lzma2 data, uncompressed bytes, header kwargs); index: records to write instead of the real ones"""
    fl = bytes([0, check]) if flags is None else flags
    out = bytearray(b"\xfd7zXZ\x00" + fl + struct.pack("<I", zlib.crc32(fl)))
    recs = []
    for data, unc, kw in blocks:
        kw = dict(kw)
        if kw.pop("sizes", False):
            kw["comp"], kw["unc"] = len(data), len(unc)
        h = block_header(**kw)
        blk = h + data
        blk += bytes(-len(blk) % 4)
        ck = check_field(check, unc)
        recs.append((len(h) + len(data) + len(ck), len(unc)))
        out += blk + ck
    recs = recs if index is None else index
    idx = b"\x00" + vli(len(recs)) + b"".join(vli(a) + vli(b) for a, b in recs)
    idx += bytes(-len(idx) % 4)
    idx += struct.pack("<I", zlib.crc32(idx))
    out += idx
    tail = struct.pack("<I", len(idx) // 4 - 1) + fl
    out += struct.pack("<I", zlib.crc32(tail)) + tail + b"YZ"
    return bytes(out)


def chunks_of(raw: bytes):
    """-> [(offset, control, header length, total length)] of the LZMA2 chunks of raw LZMA2 data"""
    out, p = [], 0
    while raw[p]:
        c = raw[p]
        if c >= 0x80:
            hl = 6 if c >= 0xC0 else 5
            tl = hl + (raw[p + 3] << 8) + raw[p + 4] + 1
        else:
            hl = 3
            tl = hl + (raw[p + 1] << 8) + raw[p + 2] + 1
        out.append((p, c, hl, tl))
        p += tl
    return out


# ---------------------------------------------------------------------------------------------------- liblzma's verdict
def liblzma_verdict(payload: bytes) -> str:
    """"ok" / "truncated" / "rejected" / "unsupported" from `xz -t` (or, without xz, from lzma for a single stream)"""
    if XZ:
        r = subprocess.run([XZ, "-t", "-q", "-q", "--format=xz", "-"], input=payload, capture_output=True)
        if r.returncode == 0:
            return "ok"
        r = subprocess.run([XZ, "-t", "--format=xz", "-"], input=payload, capture_output=True)
        msg = r.stderr.decode(errors="replace")
        if "Unexpected end of input" in msg:
            return "truncated"
        if "Unsupported" in msg:
            return "unsupported"
        return "rejected"
    d = lzma.LZMADecompressor(lzma.FORMAT_XZ)
    try:
        d.decompress(payload)
    except lzma.LZMAError as e:
        return "unsupported" if "nsupported" in str(e) else "rejected"
    if not d.eof:
        return "truncated"
    return "ok" if not d.unused_data else "rejected"


def liblzma_decode(payload: bytes) -> bytes:
    """liblzma's bytes for a valid payload (`xz -dc` reads stream padding and concatenated streams; lzma.decompress stops at
    padding)"""
    if XZ:
        return subprocess.run([XZ, "-dc", "--format=xz", "-"], input=payload, capture_output=True, check=True).stdout
    return lzma.decompress(payload)


def src_text(n, seed=1):
    return synth.jsonlog_text(n, seed)


# ---------------------------------------------------------------------------------------------------- cases
def valid_cases():
    """-> [(name, payload, data)]: payloads liblzma accepts, with their decoded bytes"""
    t = src_text(200000)
    rnd = random.Random(5).randbytes(150000)
    cases = []
    for p in list(range(10)) + [9 | lzma.PRESET_EXTREME, 6 | lzma.PRESET_EXTREME]:
        d = t[: 20000 + 15000 * (p & 15)]
        cases.append((f"preset{p}", lzma.compress(d, preset=p), d))
    for lc, lp, pb in [(0, 0, 0), (3, 0, 2), (0, 4, 0), (4, 0, 4), (1, 3, 2), (2, 2, 1), (3, 1, 0), (4, 0, 0)]:
        f = [{"id": lzma.FILTER_LZMA2, "preset": 6, "lc": lc, "lp": lp, "pb": pb}]
        cases.append((f"lclppb{lc}{lp}{pb}", lzma.compress(t[:60000], filters=f), t[:60000]))
    for ds in [4096, 1 << 16, 3 << 20, 64 << 20]:
        f = [{"id": lzma.FILTER_LZMA2, "preset": 6, "dict_size": ds}]
        cases.append((f"dict{ds}", lzma.compress(t, filters=f), t))
    for ck in [lzma.CHECK_NONE, lzma.CHECK_CRC32, lzma.CHECK_CRC64, lzma.CHECK_SHA256]:
        cases.append((f"check{ck}", lzma.compress(t[:50000], check=ck), t[:50000]))
    mix = rnd[:70000] + t[:40000] + rnd[70000:] + t[40000:90000]
    cases.append(("random", lzma.compress(rnd), rnd))
    cases.append(("random_text", lzma.compress(mix), mix))
    cases.append(("empty", lzma.compress(b""), b""))
    cases.append(("one_byte", lzma.compress(b"x"), b"x"))
    # raw LZMA2 pieces concatenated without their end byte: a dictionary reset in the middle of a block
    pieces = [t[:30000], rnd[:20000], t[30000:90000], b"z" * 5000]
    raw = b"".join(raw_lzma2(p)[:-1] for p in pieces) + b"\x00"
    d = b"".join(pieces)
    cases.append(("midblock_reset", stream([(raw, d, {})], check=1), d))
    # multi-block, by hand: with and without sizes in the block headers, every check type
    for ck in (0, 1, 4, 10):
        bl = [(raw_lzma2(p, preset=1), p, {"sizes": bool(i & 1), "dict_code": 16 + i}) for i, p in enumerate(pieces)]
        cases.append((f"blocks_check{ck}", stream(bl, check=ck), d))
    # blocks without chunks (LZMA2 data = the end byte alone), in the middle of a stream with and without sizes in the header,
    # first in a stream, and last in a stream that another stream follows: the segment around them spans them
    a, b = t[:5000], t[5000:9000]
    ra, rb = raw_lzma2(a), raw_lzma2(b)
    for sz in (False, True):
        cases.append((f"empty_block_mid{int(sz)}", stream([(ra, a, {}), (b"\x00", b"", {"sizes": sz}), (rb, b, {})]), a + b))
    cases.append(("empty_blocks_first", stream([(b"\x00", b"", {}), (b"\x00", b"", {"sizes": True}), (ra, a, {})], check=4), a))
    cases.append(("empty_block_then_stream", stream([(ra, a, {}), (b"\x00", b"", {})], check=0) + bytes(4) +
                  stream([(b"\x00", b"", {}), (rb, b, {})], check=1), a + b))
    # concatenated streams with stream padding
    s1, s2, s3 = lzma.compress(t[:10000]), lzma.compress(rnd[:3000], check=lzma.CHECK_NONE), lzma.compress(b"")
    cases.append(("concat", s1 + s2, t[:10000] + rnd[:3000]))
    cases.append(("concat_pad", s1 + bytes(8) + s2 + bytes(4) + s3 + bytes(12), t[:10000] + rnd[:3000]))
    cases.append(("trailing_pad", s1 + bytes(4), t[:10000]))
    if XZ:
        big = src_text(600000, 7)
        r = subprocess.run([XZ, "-T2", "--block-size=65536", "-c", "-6"], input=big, capture_output=True, check=True)
        cases.append(("xz_T2_blocks", r.stdout, big))
        r = subprocess.run([XZ, "-c", "-0", "--check=sha256"], input=big[:100000], capture_output=True, check=True)
        cases.append(("xz_cli", r.stdout, big[:100000]))
    return cases


def _flip(b: bytes, i: int, mask=1) -> bytes:
    x = bytearray(b)
    x[i] ^= mask
    return bytes(x)


def invalid_cases():
    """-> [(name, payload, cap, expected xzref verdict)]"""
    t = src_text(40000, 3)
    rnd = random.Random(9).randbytes(20000)
    cases = []
    small = stream([(raw_lzma2(t[:300], preset=1), t[:300], {"sizes": True}), (raw_lzma2(rnd[:50]), rnd[:50], {})], check=1)
    n_small = 350
    for cut in range(len(small)):
        cases.append((f"trunc{cut}", small[:cut], n_small, None))
    # header CRCs
    bh = 12   # block header of the first block
    hs = (small[bh] + 1) * 4
    cases.append(("crc_stream_header", _flip(small, 8), n_small, "data"))
    cases.append(("crc_block_header", _flip(small, bh + hs - 1), n_small, "data"))
    cases.append(("crc_index", _flip(small, len(small) - 13), n_small, "data"))
    cases.append(("crc_footer", _flip(small, len(small) - 12), n_small, "data"))
    cases.append(("footer_magic", _flip(small, len(small) - 1), n_small, "data"))
    cases.append(("footer_backward_size", _flip(small, len(small) - 8, 1), n_small, "data"))
    # index against the blocks
    p1, p2 = raw_lzma2(t[:1000]), raw_lzma2(t[1000:3000])
    bl = [(p1, t[:1000], {}), (p2, t[1000:3000], {})]
    good = stream(bl, check=0)
    hl = len(block_header())
    cases.append(("index_count", stream(bl, check=0, index=[(hl + len(p1), 1000)]), 3000, "data"))
    cases.append(("index_unpacked", stream(bl, check=0, index=[(hl + len(p1), 1000), (hl + len(p2), 2001)]), 3000, "data"))
    recs = [(hl + len(p1), 1000), (hl + len(p2), 2000)]
    cases.append(("index_swapped", stream(bl, check=0, index=recs[::-1]), 3000, "data"))
    cases.append(("index_unpadded", stream(bl, check=0, index=[(hl + len(p1) + 1, 1000), (hl + len(p2), 2000)]), 3000, "data"))
    cases.append(("block_header_sizes", stream([(p1, t[:1000], {"comp": len(p1) + 1})], check=0), 1000, "data"))
    cases.append(("block_header_unc", stream([(p1, t[:1000], {"unc": 999})], check=0), 1000, "data"))
    # stream padding
    for k in (1, 2, 3, 5):
        cases.append((f"padding{k}", good + bytes(k), 3000, "data"))
    cases.append(("garbage_after", good + bytes(range(1, 13)), 3000, "data"))
    # an end-of-stream marker: a raw LZMA1 stream (which always ends with one) as an LZMA2 chunk one byte longer than its data
    d = t[:3000]
    l1 = lzma.compress(d, format=lzma.FORMAT_RAW, filters=[{"id": lzma.FILTER_LZMA1, "preset": 6, "lc": 3, "lp": 0, "pb": 2}])
    u = len(d) + 1
    ch = bytes([0xE0 | ((u - 1) >> 16), ((u - 1) >> 8) & 255, (u - 1) & 255, ((len(l1) - 1) >> 8) & 255, (len(l1) - 1) & 255, 93]) + l1
    cases.append(("eos_marker", stream([(ch + b"\x00", d + b"?", {})], check=0), u, "data"))
    # lc + lp = 5 in the first chunk's properties
    raw = raw_lzma2(t[:5000])
    assert raw[0] >= 0xE0
    cases.append(("lclp5", stream([(raw[:5] + bytes([(2 * 5 + 1) * 9 + 4]) + raw[6:], t[:5000], {})], check=0), 5000, "data"))
    cases.append(("props225", stream([(raw[:5] + bytes([225]) + raw[6:], t[:5000], {})], check=0), 5000, "data"))
    # an LZMA chunk without properties after a dictionary reset (an uncompressed chunk 0x01, then 0xA0)
    noprops = b"\x01\x00\x09" + b"0123456789" + bytes([0xA0 | (raw[0] & 0x1F)]) + raw[1:5] + raw[6:]
    cases.append(("no_props_after_reset", stream([(noprops, b"0123456789" + t[:5000], {})], check=0), 5010, "data"))
    # first chunk 0x02 (no dictionary reset), and an LZMA first chunk without one (0xC0)
    cases.append(("first_chunk_02", stream([(b"\x02\x00\x03abcd\x00", b"abcd", {})], check=0), 4, "data"))
    cases.append(("first_chunk_c0", stream([(bytes([0xC0 | (raw[0] & 0x1F)]) + raw[1:], t[:5000], {})], check=0), 5000, "data"))
    cases.append(("control_03", stream([(b"\x01\x00\x03abcd\x03\x00\x00\x00", b"abcd", {})], check=0), 8, "data"))
    # a distance beyond the dictionary: X + X with X = 10,000 random bytes, encoded with a 64 KiB dictionary, declared 4 KiB
    x = rnd[:10000]
    rx = raw_lzma2(x + x, dict_size=1 << 16)
    cases.append(("distance_beyond_dict", stream([(rx, x + x, {"dict_code": 0})], check=0), 20000, "data"))
    # a distance beyond the bytes produced since the last reset: the same chunks behind a dictionary reset that cuts them
    rr = raw_lzma2(x + x, dict_size=1 << 16, preset=0)
    cs = chunks_of(rr)
    if len(cs) >= 2 and cs[1][1] & 0xE0 in (0xA0, 0xC0):
        o, c, hl2, tl = cs[1]
        props = bytes([rr[o + 5]]) if c >= 0xC0 else bytes([rr[cs[0][0] + 5]]) if cs[0][1] >= 0xC0 else bytes([93])
        cut = rr[:o] + bytes([0xE0 | (c & 0x1F)]) + rr[o + 1:o + 5] + props + rr[o + hl2:]
        cases.append(("distance_before_reset", stream([(cut, x + x, {})], check=0), 20000, "data"))
    # a range coder not finished at the end of its chunk: one byte more than its data
    pk = (raw[3] << 8) + raw[4] + 1
    longer = raw[:3] + bytes([(pk >> 8) & 255, pk & 255]) + raw[5:6 + pk - 1] + b"\x00" + raw[6 + pk - 1:]
    cases.append(("rc_not_finished", stream([(longer, t[:5000], {})], check=0), 5000, "data"))
    cases.append(("rc_corrupt", stream([(_flip(raw, 6 + pk - 2, 0x40), t[:5000], {})], check=0), 5000, "data"))
    cases.append(("rc_first_byte", stream([(_flip(raw, 6, 0x80), t[:5000], {})], check=0), 5000, "data"))
    # filters other than one LZMA2 filter: not on this path
    cases.append(("filter_delta", stream([(p1, t[:1000], {"filters": [(0x03, b"\x00")]})], check=0), 1000, "method"))
    bcj = lzma.compress(t[:8000], filters=[{"id": lzma.FILTER_X86}, {"id": lzma.FILTER_LZMA2, "preset": 1}])
    cases.append(("filter_bcj_lzma2", bcj, 8000, "method"))
    cases.append(("filter_unknown", stream([(p1, t[:1000], {"filters": [(0x7777, b"\x00")]})], check=0), 1000, "method"))
    cases.append(("block_reserved_flags", stream([(p1, t[:1000], {})], check=0).replace(b"\x00\x21\x01", b"\x04\x21\x01", 1), 1000, None))
    # a reserved check ID
    cases.append(("check_reserved", stream([(p1, t[:1000], {})], check=2, flags=b"\x00\x02"), 1000, "data"))
    # more output than the directory declares: overflow; less: short
    cases.append(("overflow", good, 2999, "overflow"))
    cases.append(("overflow_raw_chunk", stream([(b"\x01\x00\x03abcd\x00", b"abcd", {})], check=0), 3, "overflow"))
    cases.append(("short", good, 3100, "short"))
    return cases


# ---------------------------------------------------------------------------------------------------- tests
@pytest.fixture(scope="module")
def valid():
    return valid_cases()


@pytest.fixture(scope="module")
def invalid():
    return invalid_cases()


def test_valid_against_liblzma(valid):
    for name, payload, data in valid:
        assert liblzma_decode(payload) == data, name
        out, v = xzref.decode(payload, len(data))
        assert v == "ok" and out == data, (name, v)
        if XZ:
            assert liblzma_verdict(payload) == "ok", name


def test_valid_cases_cover_the_format(valid):
    """the valid cases reach uncompressed chunks, state resets, dictionary resets inside a block, and several blocks and
    streams"""
    kinds = set()
    for name, payload, data in valid:
        chunks, v = xzref.walk(payload, len(data))
        for kind, lo, pk, unp, props, reset, dsz in chunks:
            kinds.add((kind, reset))
            if props:
                kinds.add(("lclp", props[0] + props[1]))
    assert {("copy", "dict"), ("lzma", "dict"), ("lzma", None), ("lclp", 4), ("lclp", 3)} <= kinds, kinds


def test_invalid_against_liblzma(invalid):
    for name, payload, cap, want in invalid:
        out, v = xzref.decode(payload, cap)
        if want is not None:
            assert v == want, (name, v, want)
        else:
            assert v in ("data", "truncated"), (name, v)
        if v in ("short", "overflow", "method") or name == "check_reserved":
            continue   # these verdicts depend on the ZIP entry or on what this path decodes, not on the xz payload
        lv = liblzma_verdict(payload)
        assert lv != "ok", (name, v)
        if lv == "truncated" and XZ:
            assert v == "truncated", (name, v)


def test_truncation_verdicts(invalid):
    """every proper prefix of a valid payload is rejected; a cut inside the container (not inside an LZMA chunk) is a
    truncation"""
    got = {v for name, _, _, v in [(n, p, c, xzref.decode(p, c)[1]) for n, p, c, w in invalid if n.startswith("trunc")]}
    assert got <= {"data", "truncated"} and "truncated" in got


def test_method_cases_are_valid_xz(invalid):
    """the filter chains rejected as OTZ_ST_METHOD are real xz features (liblzma decodes the BCJ one)"""
    d = {n: p for n, p, c, w in invalid}
    assert lzma.decompress(d["filter_bcj_lzma2"]) == src_text(40000, 3)[:8000]


def test_xzref_positions_and_reps():
    """lp / pb > 0 and long repeats: positions count from the last dictionary reset, across chunks and blocks"""
    rnd = random.Random(3)
    d = bytes(rnd.choice(b"abcd") for _ in range(50000)) * 3
    for lc, lp, pb in [(0, 2, 2), (1, 1, 3), (0, 4, 4)]:
        f = [{"id": lzma.FILTER_LZMA2, "preset": 6, "lc": lc, "lp": lp, "pb": pb, "dict_size": 1 << 16}]
        c = lzma.compress(d, filters=f)
        assert xzref.decode(c, len(d)) == (d, "ok")
