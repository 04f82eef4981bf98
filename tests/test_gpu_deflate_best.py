"""The best DEFLATE level (OTZ_M_BEST, libzip levels 7-9; k_deflate_best): every stream decodes with zlib, the chunk
contract of the other levels holds, the ratio reaches zlib level 6 on whole entries, the output depends only on the
source, the seam rejects what it must, and the libzip calls write, seal and read such entries."""
import ctypes as C
import json
import os
import subprocess
import sys
import zipfile
import zlib

import numpy as np
import pytest

from otezip_b200 import synth
from otezip_b200.zipapi import ZipApi, ZIP_CM_DEFLATE, ZIP_EM_AES_256

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DBG = os.path.join(ROOT, "otezip_b200", "libotezip_b200_dbg.so")
BEST, FAST = 0x200, 0x100
CHUNK = 65280


def edge_sources():
    """(name, bytes) of the edge cases of the best level's search"""
    t = synth.jsonlog_text(1 << 20, 501)
    out = [("len%d" % n, t[:n]) for n in (0, 1, 2, 3, 4, 5, 257, 258, 259, 65279, 65280, 65281, 3 * 65280 + 7)]
    out += [("text1M", t), ("A200000", b"A" * 200000), ("period2", b"ab" * 40000), ("period3", b"xyz" * 30001),
            ("bytes256", bytes(range(256))), ("random", synth.random_bytes(300000, 8))]
    r = synth.random_bytes(40000, 9)
    out += [("dist32768", r[:32768] + r[:300]), ("dist32769", r[:32769] + r[:300])]
    x = synth.jsonlog_text(CHUNK, 10)   # text, so the entry is DEFLATE and chunk 2 has to decode alone
    out += [("straddle", x + x[-1000:] + synth.jsonlog_text(5000, 11))]   # chunk 2 begins with a copy of chunk 1's end
    out += [("collide", hash_collisions())]
    return out


def hash_collisions():
    """words that share the 14-bit hash of the best level (and the 9-bit one of the default level), in a random order with
    repeats, so chains are long and full of strangers"""
    rng = np.random.default_rng(12)
    v = rng.integers(0, 1 << 32, size=1 << 23, dtype=np.uint64)
    h = ((v * 2654435761) & 0xFFFFFFFF) >> 18
    words = v[h == 77].astype(np.uint32)[:256]
    assert len(words) >= 64
    seq = words[rng.integers(0, len(words), size=60000)]
    return seq.astype("<u4").tobytes()


def c5_slice():
    pool = synth.TextPool(64 << 20, seed=5)
    offs = pool.offsets([262144] * 32)
    return [pool.at(offs[i], 262144) for i in range(32)]


def zlib_raw(s, level):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return c.compress(s) + c.flush()


def run_job(ctx, srcs, methods):
    """the device-resident seam: -> (payloads, method_out, crc, first_chunk, n_chunks, csize)"""
    n = len(srcs)
    lens = np.array([len(s) for s in srcs], dtype=np.uint32)
    ofs = np.zeros(n, dtype=np.uint64)
    pos = 0
    for i in range(n):
        ofs[i] = pos
        pos += (int(lens[i]) + 15) & ~15
    img = np.zeros(max(pos, 1), dtype=np.uint8)
    for i, s in enumerate(srcs):
        img[int(ofs[i]):int(ofs[i]) + len(s)] = np.frombuffer(s, dtype=np.uint8)
    d_in = ctx.dev_alloc(img.nbytes)
    ctx.h2d(d_in, img)
    job = ctx.deflate_plan(ofs, lens, np.array(methods, dtype=np.uint16))
    try:
        ctx.deflate_run(job, d_in, img.nbytes)
        o, sz, crc, mo, total = ctx.deflate_results(job, n)
        out = ctx.deflate_fetch(job, total)
        first, cnt, cs, cb = ctx.deflate_chunks(job, n)
        assert cb == CHUNK
    finally:
        ctx.deflate_destroy(job)
        ctx.dev_free(d_in)
    pays = [bytes(out[int(o[i]):int(o[i]) + int(sz[i])]) for i in range(n)]
    return pays, [int(m) for m in mo], [int(c) for c in crc], first, cnt, cs


@pytest.fixture(scope="module")
def edges():
    return edge_sources()


def test_best_roundtrip_edge_sources(ctx, edges):
    srcs = [s for _, s in edges]
    best = ctx.deflate_host(srcs, [8 | BEST] * len(srcs))
    dflt = ctx.deflate_host(srcs, [8] * len(srcs))
    for (name, s), (m, p, crc), (md, pd, _) in zip(edges, best, dflt):
        assert crc == zlib.crc32(s) & 0xFFFFFFFF, name
        if m == 8:
            assert len(p) < len(s) and zlib.decompress(p, -15) == s, name
        else:
            assert m == 0 and p == s, name   # empty, or a stream that is not smaller: STORE
        if name in ("len0", "random", "dist32769"):
            assert m == md == 0, name        # the STORE fallback, as at the default level
    got = dict(zip([n for n, _ in edges], best))
    assert got["dist32768"][0] == 8 and len(got["dist32768"][1]) < 33068 - 200   # the repeat at exactly 32,768 is used
    assert got["A200000"][0] == 8 and len(got["A200000"][1]) < 1000


def test_best_chunk_contract(ctx, edges):
    srcs = [s for _, s in edges]
    pays, mo, _, first, cnt, cs = run_job(ctx, srcs, [8 | BEST] * len(srcs))
    for i, (name, s) in enumerate(edges):
        if mo[i] != 8:
            continue
        pos = 0
        for k in range(int(cnt[i])):
            b = pays[i][pos:pos + int(cs[int(first[i]) + k])]
            pos += len(b)
            d = zlib.decompressobj(-15)
            piece = d.decompress(b)   # alone: no reference into an earlier chunk
            assert piece == s[k * CHUNK:(k + 1) * CHUNK], (name, k)
            last = k + 1 == int(cnt[i])
            assert d.eof == last and not d.unused_data, (name, k)   # BFINAL only on the last chunk
            if ((b[0] >> 1) & 3) == 0:
                assert len(b) == 5 + len(piece), (name, k)              # one stored block: ends with the chunk's bytes
            else:
                assert b[-4:] == b"\x00\x00\xff\xff", (name, k)     # byte-aligned behind an empty stored block
        assert pos == len(pays[i]), name


def test_best_ratio_reaches_zlib6(ctx):
    srcs = c5_slice()
    best = ctx.deflate_host(srcs, [8 | BEST] * len(srcs))
    dflt = ctx.deflate_host(srcs, [8] * len(srcs))
    tot = sum(len(s) for s in srcs)
    b = d = 0
    for s, (m, p, _), (md, pd, _) in zip(srcs, best, dflt):
        assert m == 8 and zlib.decompress(p, -15) == s
        assert len(p) <= len(pd)
        b += len(p)
        d += len(pd)
    z6 = sum(len(zlib_raw(s, 6)) for s in srcs)
    z9 = sum(len(zlib_raw(s, 9)) for s in srcs)
    print("c5 slice ratio: best %.3f  default %.3f  zlib-6 %.3f  zlib-9 %.3f" % (tot / b, tot / d, tot / z6, tot / z9))
    assert tot / b >= tot / z6


def test_best_is_deterministic(ctx, edges):
    srcs = [s for _, s in edges] + c5_slice()[:6]
    a = run_job(ctx, srcs, [8 | BEST] * len(srcs))[0]
    b = run_job(ctx, srcs, [8 | BEST] * len(srcs))[0]
    assert a == b
    perm = list(range(len(srcs)))[::-1]
    perm = perm[1::2] + perm[0::2]
    # another order, and best entries mixed with default / fast / STORE ones in the same job
    extra = [synth.jsonlog_text(100000, 77)] * 3
    order = [srcs[i] for i in perm] + extra
    meths = [8 | BEST] * len(srcs) + [8, 8 | FAST, 0]
    c = run_job(ctx, order, meths)[0]
    for k, i in enumerate(perm):
        assert c[k] == a[i], i
    alone = [ctx.deflate_host([extra[0]], [m])[0][1] for m in (8, 8 | FAST)]
    assert c[-3:] == alone + [extra[0]]


def test_best_plan_rejects_bad_levels(ctx):
    L = ctx.lib.L
    for meth in (0x308, 0x200 | 93, 0x200):
        ofs = np.zeros(1, dtype=np.uint64)
        ln = np.full(1, 100, dtype=np.uint32)
        m = np.full(1, meth, dtype=np.uint16)
        j = C.c_void_p()
        rc = L.otz_deflate_plan(ctx.h, ofs.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p), m.ctypes.data_as(C.c_void_p), 1,
                                C.byref(j))
        assert rc == -2 and not j.value, hex(meth)
        assert b"otz_deflate_plan" in L.otz_last_error()


def test_best_through_libzip_api(tmp_path, refread):
    from tests.test_gpu_aes import read as aes_read, _write as aes_write, PW
    api = ZipApi()
    data = [("big.json", synth.jsonlog_text(3 << 20, 61)), ("mid.json", synth.jsonlog_text(200000, 62)),
            ("small.json", synth.jsonlog_text(3000, 63)), ("rand.bin", synth.random_bytes(100000, 64)), ("empty", b"")]
    want = [d for _, d in data]

    def payloads(p):
        with zipfile.ZipFile(p) as z:
            raw = open(p, "rb").read()
            pays = []
            for inf in z.infolist():
                nl, xl = np.frombuffer(raw[inf.header_offset + 26:inf.header_offset + 30], dtype="<u2")
                o = inf.header_offset + 30 + int(nl) + int(xl)
                pays.append(raw[o:o + inf.compress_size])
            if not any(inf.flag_bits & 1 for inf in z.infolist()):
                assert [z.read(inf) for inf in z.infolist()] == [d for d in want[:len(pays)]]
        return pays

    def write(name, level):
        p = str(tmp_path / name)
        if level is None:   # zip_set_file_compression never called: the archive's default method, no level
            assert api.write_archive(p, [(n, d) for n, d in data], ZIP_CM_DEFLATE, use_default_method=True) == 0
        else:
            assert api.write_archive(p, [(n, d, ZIP_CM_DEFLATE, level) for n, d in data]) == 0
        return p, payloads(p)

    paths, pays = {}, {}
    for lvl in (None, 0, 6, 7, 8, 9):
        paths[lvl], pays[lvl] = write("l%s.zip" % lvl, lvl)
    assert pays[7] == pays[8] == pays[9]
    assert pays[0] == pays[6] == pays[None]
    assert len(pays[9][0]) < len(pays[None][0])
    err, names, datas = api.read_all(paths[9])        # multi-chunk entries take the chunk index
    assert err == 0 and datas == want
    e2, got = refread.extract_file(paths[9], verify_crc=1)
    assert e2 == 0 and got == want
    # AES-256 at level 9: the sealed payload is the best-level stream plus salt (16), verifier (2) and code (10)
    p = tmp_path / "aes9.zip"
    assert aes_write(api, p, [("b.json", want[0], ZIP_CM_DEFLATE, 9, 0), ("s.json", want[1], ZIP_CM_DEFLATE, 9, ZIP_EM_AES_256)]) == 0
    res = aes_read(api, p, PW)
    assert [r[0] for r in res] == [want[0], want[1]]
    pa = payloads(str(p))
    assert pa[0] == pays[9][0] and len(pa[1]) == len(pays[9][1]) + 28 and len(pays[9][1]) < len(pays[None][1])


CHILD = r'''
import ctypes as C, json, sys, zlib
sys.path.insert(0, %(root)r)
from otezip_b200 import Ctx
from otezip_b200.native import Lib
from tests.test_gpu_deflate_best import edge_sources, c5_slice
L = Lib.get().L
L.otz_debug_violations.argtypes = [C.c_void_p, C.c_int]
c = Ctx(0)
srcs = [s for _, s in edge_sources()] + c5_slice()
bad = 0
for s, (m, p, crc) in zip(srcs, c.deflate_host(srcs, [8 | 0x200] * len(srcs))):
    if (zlib.decompress(p, -15) if m == 8 else p) != s or crc != (zlib.crc32(s) & 0xFFFFFFFF):
        bad += 1
c.close()
v = (C.c_uint64 * 32)()
n = L.otz_debug_violations(v, 32)
print(json.dumps({"slots": n, "violations": [int(x) for x in v[:max(n, 0)]], "mismatches": bad, "sources": len(srcs)}))
'''


@pytest.mark.skipif(not os.path.exists(DBG), reason="debug library not built (make debug)")
def test_best_bounds_checked_build():
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}], capture_output=True, text=True, timeout=1200, cwd=ROOT,
                       env=dict(os.environ, OTEZIP_B200_LIB=DBG))
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["slots"] > 0, "the debug library must have the checks compiled in"
    assert d["mismatches"] == 0 and sum(d["violations"]) == 0, d
