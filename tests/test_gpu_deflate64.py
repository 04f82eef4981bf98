"""Deflate64 entries (ZIP method 9) on the GPU, against the plain-Python decoder of tests/deflate64.py: bytes, status class and
produced length, through every (lanes, ring) instantiation, the C-ABI host calls and the libzip-subset API."""
import ctypes as C
import json
import os
import random
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

from otezip_b200 import Ctx, synth
from otezip_b200.native import Lib, parse_central, default_opts
from otezip_b200.zipapi import ZipApi, ZIP_CREATE, ZIP_TRUNCATE
from tests import aeszip
from tests.deflate64 import inflate, Encoder
from tests.test_deflate64_cpu import KA, KA_BAD, BitW, fixed_lit
from tests.test_gpu_inflate_configs import CONFIGS

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFDIR = os.path.join(ROOT, "oracle", "_ref")
ST_OK, ST_DATA, ST_TRUNC, ST_OVER, ST_METHOD = 0, 7, 8, 9, 5
F_CRC, F_REF, F_SHORT = 0x100, 0x200, 0x400
VERDICT = {"ok": ST_OK, "short": ST_OK, "data": ST_DATA, "truncated": ST_TRUNC, "overflow": ST_OVER}


def build(members, zip64=False):
    """members: (name, method, payload, uncomp_size, crc).  Four zero bytes follow every payload, so that the bits a decoder
    reads past the end of a truncated stream are zero wherever the image lands (as tests/deflate64.py reads them)."""
    out, cd = bytearray(), bytearray()
    for name, m, p, u, crc in members:
        nm = name.encode()
        ofs = len(out)
        out += struct.pack("<IHHHHHIIIHH", 0x04034B50, 20, 0, m, 0, 0x21, crc, len(p), u, len(nm), 0) + nm + p + bytes(4)
        cd += struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, 0x031E, 20, 0, m, 0, 0x21, crc, len(p), u, len(nm), 0, 0, 0, 0,
                          0o100644 << 16, ofs) + nm
    n, cdo = len(members), len(out)
    out += cd
    if zip64:
        r = len(out)
        out += struct.pack("<IQHHIIQQQQ", 0x06064B50, 44, 45, 45, 0, 0, n, n, len(cd), cdo)
        out += struct.pack("<IIQI", 0x07064B50, 0, r, 1)
        out += struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, 0xFFFF, 0xFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0)
    else:
        out += struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, n, n, len(cd), cdo, 0)
    return bytes(out)


def extract(img, env=None):
    """-> (arena, table, crc, status, produced) through otz_extract_host_ex"""
    env = env or {}
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        c = Ctx(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    tab = parse_central(img)
    n = len(tab)
    out_len = int((tab["out_ofs"].astype(np.int64) + tab["uncomp_size"]).max()) if n else 0
    out = np.zeros(max(out_len, 1), np.uint8)
    crc, st, prod = np.zeros(max(n, 1), np.uint32), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.uint32)
    buf = np.frombuffer(img, np.uint8)
    L = c.L
    vp = C.c_void_p
    L.otz_extract_host_ex.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint32, vp, vp, C.c_uint64, vp, vp, vp]
    o = default_opts()
    c.lib.check(L.otz_extract_host_ex(c.h, buf.ctypes.data, buf.nbytes, np.ascontiguousarray(tab).ctypes.data, n, C.byref(o),
                                      out.ctypes.data, out_len, crc.ctypes.data, st.ctypes.data, prod.ctypes.data), "extract")
    c.close()
    return out, tab, crc[:n], st[:n], prod[:n]


_REF = {}


def reference(p, u):
    k = (zlib.crc32(p), len(p), u)
    if k not in _REF:
        _REF[k] = inflate(p, u)
    return _REF[k]


def check(members, env=None, zip64=False):
    """every method-9 member against the Python decoder; returns the GPU results"""
    img = build(members, zip64)
    out, tab, crc, st, prod = extract(img, env)
    for i, (name, m, p, u, c) in enumerate(members):
        s = int(st[i])
        if m != 9:
            continue
        exp, v = reference(p, u)
        o = int(tab["out_ofs"][i])
        assert s & 0xFF == VERDICT[v], (name, hex(s), v)
        assert int(prod[i]) == len(exp), (name, int(prod[i]), len(exp), v)
        if v in ("ok", "short"):
            assert s & F_REF and bool(s & F_SHORT) == (v == "short"), (name, hex(s))
            assert out[o:o + u].tobytes() == exp + bytes(u - len(exp)), name
            assert bool(s & F_CRC) == (int(crc[i]) != c) and int(crc[i]) == zlib.crc32(exp + bytes(u - len(exp))), name
    return img, out, tab, crc, st, prod


def member9(name, data, stream=None, mode="deflate64", block="dynamic"):
    p = stream if stream is not None else ENC().compress(data, mode, block)
    return (name, 9, p, len(data), zlib.crc32(data))


_ENC = []


def ENC():
    if not _ENC:
        _ENC.append(Encoder())
    return _ENC[0]


def corpus(seed=11):
    """seeded native Deflate64 entries: 0 B .. ~4 MiB, text and random, >= 1 MiB, matches mostly beyond 32 KiB"""
    rnd = random.Random(seed)
    pool = synth.TextPool(8 << 20, seed)
    ms = [member9("empty", b""), member9("one", b"x")]
    for i in range(40):
        n = int(2 ** rnd.uniform(0, 22))
        d = pool.take(n) if i % 3 else synth.random_bytes(n, i)
        ms.append(member9("c%02d" % i, d, block=("dynamic", "fixed", "stored", "mixed")[i % 4] if n < 300000 else "dynamic"))
    ms.append(member9("big_text", pool.take(3 << 20)))
    ms.append(member9("big_mixed", pool.take(1 << 20) + synth.random_bytes(300000, 5) + pool.take(1 << 20)))
    blob = synth.random_bytes(45000, 6)
    far = b"".join(blob[k:] + blob[:k] for k in (0, 7, 19)) * 6   # every repeat 45,000 bytes back
    ms.append(member9("far", far))
    ms.append(member9("runs", b"".join(bytes([rnd.randrange(256)]) * rnd.randint(1, 25000) for _ in range(40))))   # (under the zip-bomb ratio)
    ms.append(member9("ab", b"ab" * 150000 + b"c" * 70000))
    for name, stream, exp in KA:
        ms.append(("ka_" + name, 9, stream, len(exp), zlib.crc32(exp)))
    return ms


@pytest.fixture(scope="module")
def corpus_members():
    return corpus()


def test_corpus_and_known_answers(corpus_members):
    check(corpus_members)


@pytest.mark.parametrize("g,w", CONFIGS)
def test_every_instantiation(g, w, corpus_members):
    check(corpus_members[::3] + corpus_members[-len(KA) - 4:], {"OTZ_INFLATE_TILE": str(g), "OTZ_INFLATE_RING": str(w)})


def test_errors_and_short_streams():
    ms = []
    ka = {k[0]: k for k in KA}
    s, exp = ka["len65538_dist1"][1], ka["len65538_dist1"][2]
    d = ka["dist30_31_stored"]
    ms.append(("bad_dist", 9, KA_BAD, 100, 0))
    ms.append(("over_long_match", 9, s, len(exp) - 1, 0))
    ms.append(("over_stored", 9, d[1], 1000, 0))
    ms.append(("short", 9, s, len(exp) + 4000, zlib.crc32(exp + bytes(4000))))
    for cut in (1, 2, 3, 5, len(s) - 1):
        ms.append(("cut%d" % cut, 9, s[:cut], len(exp), 0))
    for cut in (70000, len(d[1]) - 3):
        ms.append(("dcut%d" % cut, 9, d[1][:cut], len(d[2]), 0))
    txt = synth.jsonlog_text(300000, 3)
    z = ENC().compress(txt)
    for cut in (len(z) // 2, len(z) - 2):
        ms.append(("zcut%d" % cut, 9, z[:cut], len(txt), 0))
    for sym in (286, 287):
        w = BitW().bits(1, 1).bits(1, 2)
        fixed_lit(w, ord("a"))
        fixed_lit(w, sym)
        ms.append(("sym%d" % sym, 9, w.done(), 10, 0))
    ms.append(("hlit287", 9, BitW().bits(1, 1).bits(2, 2).bits(30, 5).bits(0, 5).bits(0, 4).done() + bytes(8), 10, 0))
    ms.append(("btype3", 9, b"\x07\x00", 10, 0))
    ms.append(("empty_stream", 9, b"", 10, 0))
    img, out, tab, crc, st, prod = check(ms)
    codes = {m[0]: int(st[i]) for i, m in enumerate(ms)}
    assert codes["bad_dist"] & 0xFF == ST_DATA and codes["over_long_match"] & 0xFF == ST_OVER and codes["short"] == ST_OK | F_REF | F_SHORT
    assert codes["sym286"] & 0xFF == codes["sym287"] & 0xFF == codes["hlit287"] & 0xFF == ST_DATA


def test_dual_format_streams_and_zlib_258_matches():
    """identical bytes as method 8 and 9 decode alike; zlib streams with length-258 matches stored as method 9 decode as
    Deflate64 (i.e. differently), exactly as the Python decoder says"""
    rnd = random.Random(5)
    pool = synth.TextPool(8 << 20, 9)
    dual, m8 = [], []
    for i in range(30):
        n = int(2 ** rnd.uniform(4, 21))
        d = pool.take(n) if i % 4 else synth.random_bytes(n, i)
        p = ENC().compress(d, "dual", ("dynamic", "fixed", "mixed")[i % 3])
        dual.append(("d%02d" % i, 9, p, n, zlib.crc32(d)))
        m8.append(("d%02d" % i, 8, p, n, zlib.crc32(d)))
    img9, o9, t9, c9, s9, _ = check(dual)
    for env in ({}, {"OTZ_INFLATE_MODE": "legacy"}):
        o8, t8, c8, s8, _ = extract(build(m8), env)
        for i, m in enumerate(dual):
            u, a, b = m[3], int(t9["out_ofs"][i]), int(t8["out_ofs"][i])
            assert s9[i] & 0xFF == s8[i] & 0xFF == 0 and c9[i] == c8[i] == m[4], (m[0], hex(int(s9[i])), hex(int(s8[i])))
            assert o9[a:a + u].tobytes() == o8[b:b + u].tobytes()
    zl = []
    for i, (lvl, st_) in enumerate([(9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_RLE), (1, zlib.Z_FIXED), (9, zlib.Z_FILTERED)]):
        d = b"y" * 5000 + synth.jsonlog_text(20000, i) + b"z" * 3000
        co = zlib.compressobj(lvl, zlib.DEFLATED, -15, 8, st_)
        z = co.compress(d) + co.flush()
        zl.append(("zl%d" % i, 9, z, len(d), zlib.crc32(d)))
        assert inflate(z, len(d)) != (d, "ok")   # the stream means something else as Deflate64
    check(zl)


def test_mixed_archive_leaves_other_methods_unchanged(corpus_members):
    from tests import cases
    others = [(m.name, m.method, m.payload, m.uncomp_size, m.crc32) for m in cases.mixed_archive(seed=8, n_tiny=60, n_mid=20, n_z=4, n_s=4)]
    nine = corpus_members[::4]
    mixed = []
    for i, m in enumerate(others):
        mixed.append(m)
        if i < len(nine):
            mixed.append(nine[i])
    _, o1, t1, c1, s1, p1 = check(mixed)
    o2, t2, c2, s2, p2 = extract(build(others))
    j = 0
    for i, m in enumerate(mixed):
        if m[1] == 9:
            continue
        a, b, u = int(t1["out_ofs"][i]), int(t2["out_ofs"][j]), m[3]
        assert (int(s1[i]), int(c1[i]), int(p1[i])) == (int(s2[j]), int(c2[j]), int(p2[j])), m[0]
        assert o1[a:a + u].tobytes() == o2[b:b + u].tobytes(), m[0]
        j += 1


# ---------------------------------------------------------------- the public API

def _read(api, path, pw=None, ref_compat=1, verify_crc=0):
    api.ref_compat.value, api.verify_crc.value = ref_compat, verify_crc
    err = C.c_int(-1)
    za = api.L.zip_open(str(path).encode(), 0, C.byref(err))
    assert za, err.value
    if pw:
        api.L.zip_set_default_password(za, pw)
    res = []
    for i in range(api.L.zip_get_num_files(za)):
        zf = api.L.zip_fopen_index(za, i, 0)
        st = api.L.otezip_b200_entry_status(za, i)
        res.append((C.string_at(zf.contents.data, zf.contents.size) if zf else None, st))
        if zf:
            api.L.zip_fclose(zf)
    api.L.zip_close(za)
    return res


@pytest.fixture(scope="module")
def api():
    a = ZipApi()
    yield a
    a.ref_compat.value, a.verify_crc.value = 1, 0


def _api_members():
    pool = synth.TextPool(4 << 20, 3)
    ds = [b"", b"hello", pool.take(200000), synth.random_bytes(70000, 1), pool.take(1500000)]
    ms = [member9("f%d" % i, d) for i, d in enumerate(ds)]
    ms.append(("plain", 8, synth.deflate_raw(ds[2]), len(ds[2]), zlib.crc32(ds[2])))
    return ms, ds + [ds[2]]


def test_library_read_path(api, tmp_path):
    ms, ds = _api_members()
    p = tmp_path / "d64.zip"
    p.write_bytes(build(ms))
    r1 = _read(api, p, ref_compat=1)
    assert [x[0] for x in r1] == [None] * 5 + [ds[5]]
    assert [x[1] for x in r1] == [ST_OK | F_REF] * 5 + [0]
    r0 = _read(api, p, ref_compat=0, verify_crc=1)
    assert [x[0] for x in r0] == ds
    # a wrong CRC: reported, fatal only under otezip_verify_crc
    bad = [(n, m, pl, u, c ^ 1) for n, m, pl, u, c in ms]
    p.write_bytes(build(bad))
    assert [x[0] for x in _read(api, p, ref_compat=0, verify_crc=0)] == ds
    r = _read(api, p, ref_compat=0, verify_crc=1)
    assert [x[0] for x in r] == [None] * 6 and all(x[1] & F_CRC for x in r)
    # ZIP64 end records
    p.write_bytes(build(ms, zip64=True))
    assert [x[0] for x in _read(api, p, ref_compat=0, verify_crc=1)] == ds


def test_aes_entry_with_inner_method_9(api, tmp_path):
    ms, ds = _api_members()
    pw = b"pw"
    ents = [aeszip.Entry(n, m, pl, u, c, 1 + i % 3, 2, pw) for i, (n, m, pl, u, c) in enumerate(ms)]
    p = tmp_path / "aes.zip"
    p.write_bytes(aeszip.build_zip(ents))
    r = _read(api, p, pw, ref_compat=0, verify_crc=1)
    assert [x[0] for x in r] == ds, [hex(x[1]) for x in r]
    r = _read(api, p, pw, ref_compat=1)
    assert [x[1] for x in r[:5]] == [ST_OK | F_REF] * 5 and [x[0] for x in r[:5]] == [None] * 5


def test_method_queries_and_writer_refusal(api, tmp_path):
    L = api.L
    assert [L.zip_compression_method_supported(m, 0) for m in (0, 8, 9, 93, 12, 14)] == [1, 1, 1, 1, 0, 0]
    assert [L.zip_compression_method_supported(m, 1) for m in (0, 8, 9, 93, 12)] == [1, 1, 0, 1, 0]
    err = C.c_int(-1)
    za = L.zip_open(str(tmp_path / "w.zip").encode(), ZIP_CREATE | ZIP_TRUNCATE, C.byref(err))
    buf = C.create_string_buffer(b"abc", 3)
    i = L.zip_file_add(za, b"a", L.zip_source_buffer(za, buf, 3, 0), 0)
    assert L.zip_set_file_compression(za, i, 9, 0) == -1
    assert L.zip_close(za) == 0


SHARD = r'''
import json, sys
sys.path.insert(0, %(root)r)
from otezip_b200.zipapi import ZipApi
from tests.test_gpu_deflate64 import _read
api = ZipApi()
print(json.dumps([[None if d is None else d.hex(), s] for d, s in _read(api, %(path)r, ref_compat=int(sys.argv[1]), verify_crc=1)]))
'''


def test_sharded_over_contexts_of_one_gpu(api, tmp_path, corpus_members):
    ms = corpus_members[:30] + [m for m in _api_members()[0]]
    p = tmp_path / "shard.zip"
    p.write_bytes(build(ms))
    want = [[None if d is None else d.hex(), s] for d, s in _read(api, p, ref_compat=0, verify_crc=1)]
    for devs in ("0,0,0", "all"):
        r = subprocess.run([sys.executable, "-c", SHARD % {"root": ROOT, "path": str(p)}, "0"], capture_output=True, text=True, timeout=600,
                           cwd=ROOT, env=dict(os.environ, OTEZIP_DEVICES=devs))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.splitlines()[-1]) == want, devs


@pytest.mark.skipif(not os.path.exists(os.path.join(REFDIR, "otezip_relinked")), reason="relinked CLI not built")
def test_reference_cli_extracts_with_ref_compat_0(tmp_path, corpus_members):
    ms, ds = _api_members()
    p = tmp_path / "cli.zip"
    p.write_bytes(build(ms))
    for env, want in (({"OTEZIP_REF_COMPAT": "0"}, True), ({}, False)):
        d = tmp_path / ("out%d" % want)
        d.mkdir()
        r = subprocess.run([os.path.join(REFDIR, "otezip_relinked"), "-x", str(p), "--verify-crc"], cwd=d, capture_output=True, text=True,
                           timeout=300, env=dict(os.environ, **env))
        got = {f: open(os.path.join(d, f), "rb").read() for f in os.listdir(d)}
        if want:
            assert r.returncode == 0 and got == {m[0]: x for m, x in zip(ms, ds)}, (r.returncode, r.stderr[-500:])
        else:
            assert got.get("f2") != ds[2]


DBG_CHILD = r'''
import ctypes as C, json, sys
sys.path.insert(0, %(root)r)
from otezip_b200.native import Lib
from tests import test_gpu_deflate64 as T
from tests.test_gpu_inflate_configs import CONFIGS
ms = T.corpus(seed=12)
T.check(ms)
for g, w in [(32, 2048), (8, 1024), (4, 1024)]:
    T.check(ms[::2], {"OTZ_INFLATE_TILE": str(g), "OTZ_INFLATE_RING": str(w)})
L = Lib.get().L
L.otz_debug_violations.argtypes = [C.c_void_p, C.c_int]
v = (C.c_uint64 * 32)()
n = L.otz_debug_violations(v, 32)
print(json.dumps({"slots": n, "violations": [int(x) for x in v[:max(n, 0)]]}))
'''


def test_bounds_checked_build_counts_no_violation():
    dbg = os.path.join(ROOT, "otezip_b200", "libotezip_b200_dbg.so")
    if not os.path.exists(dbg):
        pytest.skip("debug library not built (make debug)")
    r = subprocess.run([sys.executable, "-c", DBG_CHILD % {"root": ROOT}], capture_output=True, text=True, timeout=1800, cwd=ROOT,
                       env=dict(os.environ, OTEZIP_B200_LIB=dbg))
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["slots"] > 0 and sum(d["violations"]) == 0, d
