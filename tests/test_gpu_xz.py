"""XZ entries (ZIP method 95) on the GPU, against the plain-Python decoder of tests/xzref.py and the sources: bytes, status
class and produced length through the C-ABI host call, and the libzip-subset API."""
import ctypes as C
import json
import lzma
import os
import random
import subprocess
import sys
import zlib

import numpy as np
import pytest

from otezip_b200 import synth
from otezip_b200.zipapi import ZipApi, ZIP_CREATE, ZIP_TRUNCATE, ZIP_CM_XZ
from tests import aeszip, xzref
from tests.test_gpu_deflate64 import build, extract, member9, _read, REFDIR
from tests.test_xz_cpu import valid_cases, invalid_cases, raw_lzma2, stream, liblzma_verdict

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ST_OK, ST_DATA, ST_TRUNC, ST_OVER, ST_METHOD = 0, 7, 8, 9, 5
F_CRC, F_REF, F_SHORT = 0x100, 0x200, 0x400
VERDICT = {"ok": ST_OK, "short": ST_OK, "data": ST_DATA, "truncated": ST_TRUNC, "overflow": ST_OVER, "method": ST_METHOD}


def member95(name, data, payload=None, cap=None, crc=None):
    p = payload if payload is not None else lzma.compress(data)
    return (name, 95, p, len(data) if cap is None else cap, zlib.crc32(data) if crc is None else crc)


def check(members, env=None):
    """every method-95 member against xzref; returns the GPU results"""
    img = build(members)
    out, tab, crc, st, prod = extract(img, env)
    for i, (name, m, p, u, c) in enumerate(members):
        if m != 95:
            continue
        s = int(st[i])
        want, v = xzref.decode(p, u)
        assert s & 0xFF == VERDICT[v], (name, hex(s), v)
        assert int(prod[i]) == len(want), (name, int(prod[i]), len(want), v)   # the bytes produced before the verdict
        if v in ("ok", "short"):
            a = int(tab["out_ofs"][i])
            got = out[a:a + u].tobytes()
            assert got == want + bytes(u - len(want)), name
            assert s & ~F_CRC == ST_OK | F_REF | (F_SHORT if v == "short" else 0), (name, hex(s))
            assert bool(s & F_CRC) == (zlib.crc32(got) != c), (name, hex(s))
            assert int(crc[i]) == zlib.crc32(got), name
    return img, out, tab, crc, st, prod


@pytest.fixture(scope="module")
def valid():
    return [member95(n, d, p) for n, p, d in valid_cases()]


def test_valid_payloads(valid):
    _, out, tab, crc, st, prod = check(valid)
    assert all(int(s) == ST_OK | F_REF for s in st)


def test_invalid_payloads():
    ms = [member95(n, b"", p, cap, 0) for n, p, cap, w in invalid_cases()]
    check(ms)


def test_both_shared_memory_classes_in_one_run():
    t = synth.jsonlog_text(400000, 4)
    ms = []
    for i, (lc, lp) in enumerate([(3, 0), (4, 0), (0, 4), (2, 1), (1, 3), (0, 0)] * 3):
        d = t[i * 20000:i * 20000 + 20000 + 7000 * i]
        f = [{"id": lzma.FILTER_LZMA2, "preset": 6, "lc": lc, "lp": lp, "pb": i % 5}]
        ms.append(member95("c%d" % i, d, lzma.compress(d, filters=f)))
    check(ms)


def test_many_segments():
    """16 MiB entries in 1 MiB blocks (and, in one of them, a dictionary reset every 256 KiB inside the blocks): one segment per
    block at least; entries of tiny blocks, merged into segments of at least XZ_SEG_MIN bytes across block and stream boundaries"""
    pool = synth.TextPool(40 << 20, 21)
    big = pool.take(16 << 20)
    blocks = [(raw_lzma2(big[o:o + (1 << 20)], preset=1), big[o:o + (1 << 20)], {}) for o in range(0, len(big), 1 << 20)]
    quarter = b"".join(raw_lzma2(big[o:o + (1 << 18)], preset=0)[:-1] for o in range(0, 4 << 20, 1 << 18)) + b"\x00"
    tiny = pool.take(3 << 20)
    tb = [(raw_lzma2(tiny[o:o + 5000], preset=0), tiny[o:o + 5000], {"sizes": True}) for o in range(0, len(tiny), 5000)]
    half = len(tb) // 2
    ms = [member95("blocks", big, stream(blocks, check=4)),
          member95("resets", big[:4 << 20], stream([(quarter, big[:4 << 20], {})], check=0)),
          member95("tiny_blocks", tiny, stream(tb[:half], check=1) + bytes(8) + stream(tb[half:], check=0)),
          member95("rnd", synth.random_bytes(3 << 20, 5), lzma.compress(synth.random_bytes(3 << 20, 5)))]
    check(ms)


def test_corruption_only_the_check_would_catch():
    """payloads whose LZMA data was changed so that it still decodes: liblzma rejects them by their check, this path by the ZIP
    CRC-32 -- never a clean OK"""
    d = synth.jsonlog_text(300000, 8)
    good = lzma.compress(d, check=lzma.CHECK_CRC64)
    rnd = random.Random(3)
    ms = []
    while len(ms) < 40:
        i = rnd.randrange(40, len(good) - 40)
        bad = bytearray(good)
        bad[i] ^= 1 << rnd.randrange(8)
        bad = bytes(bad)
        out, v = xzref.decode(bad, len(d))
        if v == "ok" and out != d:
            assert liblzma_verdict(bad) != "ok"
            ms.append(member95("flip%d" % i, d, bad))
        elif len(ms) < 40 and v != "ok":
            ms.append(member95("flip%d" % i, d, bad))
    _, out, tab, crc, st, prod = check(ms)
    for s in st:
        assert (int(s) & 0xFF) != ST_OK or int(s) & F_CRC


def test_mixed_archive_leaves_other_methods_unchanged(valid):
    from tests import cases
    from tests.test_gpu_deflate64 import corpus
    others = [(m.name, m.method, m.payload, m.uncomp_size, m.crc32) for m in cases.mixed_archive(seed=8, n_tiny=60, n_mid=20, n_z=4, n_s=4)]
    others += corpus(seed=13)[::6]
    assert {m[1] for m in others} >= {0, 8, 9, 93}
    mixed = []
    for i, m in enumerate(others):
        mixed.append(m)
        if i < len(valid):
            mixed.append(valid[i])
    _, o1, t1, c1, s1, p1 = check(mixed)
    o2, t2, c2, s2, p2 = extract(build(others))
    j = 0
    for i, m in enumerate(mixed):
        if m[1] == 95:
            continue
        a, b, u = int(t1["out_ofs"][i]), int(t2["out_ofs"][j]), m[3]
        assert (int(s1[i]), int(c1[i]), int(p1[i])) == (int(s2[j]), int(c2[j]), int(p2[j])), m[0]
        assert o1[a:a + u].tobytes() == o2[b:b + u].tobytes(), m[0]
        j += 1


# ---------------------------------------------------------------- the public API

@pytest.fixture(scope="module")
def api():
    a = ZipApi()
    yield a
    a.ref_compat.value, a.verify_crc.value = 1, 0


def _api_members():
    pool = synth.TextPool(4 << 20, 3)
    ds = [b"", b"hello", pool.take(200000), synth.random_bytes(70000, 1), pool.take(1500000)]
    ms = [member95("f%d" % i, d, lzma.compress(d, preset=i, check=(0, 1, 4, 10, 4)[i])) for i, d in enumerate(ds)]
    ms.append(("plain", 8, synth.deflate_raw(ds[2]), len(ds[2]), zlib.crc32(ds[2])))
    return ms, ds + [ds[2]]


def test_library_read_path(api, tmp_path, refread):
    ms, ds = _api_members()
    p = tmp_path / "xz.zip"
    p.write_bytes(build(ms))
    r1 = _read(api, p, ref_compat=1)
    assert [x[0] for x in r1] == [None] * 5 + [ds[5]]
    assert [x[1] for x in r1] == [ST_OK | F_REF] * 5 + [0]
    # the reference returns NULL for exactly these entries
    e, got = refread.extract_file(str(p), verify_crc=1)
    assert e == 0 and got == [x[0] for x in r1]
    r0 = _read(api, p, ref_compat=0, verify_crc=1)
    assert [x[0] for x in r0] == ds
    bad = [(n, m, pl, u, c ^ 1) for n, m, pl, u, c in ms]
    p.write_bytes(build(bad))
    assert [x[0] for x in _read(api, p, ref_compat=0, verify_crc=0)] == ds
    r = _read(api, p, ref_compat=0, verify_crc=1)
    assert [x[0] for x in r] == [None] * 6 and all(x[1] & F_CRC for x in r)


def test_aes_entry_with_inner_method_95(api, tmp_path):
    ms, ds = _api_members()
    pw = b"pw"
    ents = [aeszip.Entry(n, m, pl, u, c, 3, 2, pw) for n, m, pl, u, c in ms]
    p = tmp_path / "aes.zip"
    p.write_bytes(aeszip.build_zip(ents))
    r = _read(api, p, pw, ref_compat=0, verify_crc=1)
    assert [x[0] for x in r] == ds, [hex(x[1]) for x in r]
    r = _read(api, p, pw, ref_compat=1)
    assert [x[1] for x in r[:5]] == [ST_OK | F_REF] * 5 and [x[0] for x in r[:5]] == [None] * 5


def test_method_queries_and_writer_refusal(api, tmp_path):
    L = api.L
    assert ZIP_CM_XZ == 95
    assert L.zip_compression_method_supported(95, 0) == 1 and L.zip_compression_method_supported(95, 1) == 0
    err = C.c_int(-1)
    za = L.zip_open(str(tmp_path / "w.zip").encode(), ZIP_CREATE | ZIP_TRUNCATE, C.byref(err))
    buf = C.create_string_buffer(b"abc", 3)
    i = L.zip_file_add(za, b"a", L.zip_source_buffer(za, buf, 3, 0), 0)
    assert L.zip_set_file_compression(za, i, 95, 0) == -1
    assert L.zip_close(za) == 0


SHARD = r'''
import json, sys
sys.path.insert(0, %(root)r)
from otezip_b200.zipapi import ZipApi
from tests.test_gpu_deflate64 import _read
api = ZipApi()
print(json.dumps([[None if d is None else d.hex(), s] for d, s in _read(api, %(path)r, ref_compat=0, verify_crc=1)]))
'''


def test_sharded_over_contexts_of_one_gpu(api, tmp_path, valid):
    ms = valid[:30] + _api_members()[0]
    p = tmp_path / "shard.zip"
    p.write_bytes(build(ms))
    want = [[None if d is None else d.hex(), s] for d, s in _read(api, p, ref_compat=0, verify_crc=1)]
    r = subprocess.run([sys.executable, "-c", SHARD % {"root": ROOT, "path": str(p)}], capture_output=True, text=True, timeout=600,
                       cwd=ROOT, env=dict(os.environ, OTEZIP_DEVICES="0,0"))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.splitlines()[-1]) == want


@pytest.mark.skipif(not os.path.exists(os.path.join(REFDIR, "otezip_relinked")), reason="relinked CLI not built")
def test_reference_cli_extracts_with_ref_compat_0(tmp_path):
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
from tests import test_gpu_xz as T
from tests.test_xz_cpu import valid_cases, invalid_cases
T.check([T.member95(n, d, p) for n, p, d in valid_cases()])
T.check([T.member95(n, b"", p, cap, 0) for n, p, cap, w in invalid_cases()])
T.test_many_segments()
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
