"""WinZip AES entries (method 99) through the library on the GPU.  The reference is tests/aeszip.py; the specification of the
read path is the twin: with the right password an encrypted entry gives exactly what the same compressed bytes stored
unencrypted give (same bytes, same status word, same accept/reject under every switch)."""
import ctypes as C
import json
import os
import random
import struct
import subprocess
import sys
import zipfile
import zlib

import pytest

from otezip_b200 import synth
from otezip_b200.zipapi import ZipApi, ZIP_CREATE, ZIP_TRUNCATE, ZIP_EM_AES_128, ZIP_EM_AES_192, ZIP_EM_AES_256
from tests import aeszip
from tests.test_gpu_inflate_twophase import _shapes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
PW = b"correct horse battery staple"
ST_NOPASSWD, ST_WRONGPASSWD, ST_AUTH, ST_DATA_RANGE = 11, 12, 13, 3


@pytest.fixture(scope="module")
def api():
    return ZipApi()


def read(api, path, pw=None, verify_crc=0, ref_compat=1, per_entry=None):
    """-> [(bytes | None, status word)] for every entry; per_entry: {index: password} for zip_fopen_index_encrypted"""
    api.verify_crc.value = verify_crc
    api.ref_compat.value = ref_compat
    err = C.c_int(-1)
    za = api.L.zip_open(str(path).encode(), 0, C.byref(err))
    assert za, err.value
    if pw is not None:
        assert api.L.zip_set_default_password(za, pw) == 0
    res = []
    for i in range(api.L.zip_get_num_files(za)):
        if per_entry and i in per_entry:
            zf = api.L.zip_fopen_index_encrypted(za, i, 0, per_entry[i])
        else:
            zf = api.L.zip_fopen_index(za, i, 0)
        st = api.L.otezip_b200_entry_status(za, i)
        if not zf:
            res.append((None, st))
            continue
        n = zf.contents.size
        res.append((C.string_at(zf.contents.data, n) if n else b"", st))
        api.L.zip_fclose(zf)
    assert api.L.zip_close(za) == 0
    return res


def _members():
    """(name, method, payload, uncomp_size, stored crc, plaintext or None)"""
    out = []
    for m in _shapes():
        out.append((m.name, m.method, m.payload, m.uncomp_size, m.crc32, m.raw))
    for d in aeszip.read_zip(open(os.path.join(G, "edges.zip"), "rb").read()):   # every golden edge stream, as stored
        if d["method"] in (0, 8, 93):
            out.append(("edge/" + d["name"], d["method"], d["raw"], d["uncomp_size"], d["crc32"], None))
    for i, n in enumerate([0, 1, 15, 16, 17, 4096, 65535, 65536, 65537, 300001]):
        raw = synth.random_bytes(n, 60 + i)
        out.append(("store/%d" % n, 0, raw, n, zlib.crc32(raw), raw))
    try:
        from otezip_b200.zstdlib import Zstd
        zs = Zstd()
        for i, (d, lvl) in enumerate([(synth.jsonlog_text(300000, 31), 1), (synth.jsonlog_text(150000, 33), 19), (synth.random_bytes(70000, 34), 3)]):
            out.append(("zst/%d" % i, 93, zs.compress(d, lvl), len(d), zlib.crc32(d), d))
    except OSError:
        pass
    return out


@pytest.fixture(scope="module")
def twins(tmp_path_factory, api):
    d = tmp_path_factory.mktemp("aes_twins")
    ms = _members()
    plain = d / "plain.zip"
    plain.write_bytes(aeszip.build_zip([aeszip.Entry(n, m, p, u, c) for n, m, p, u, c, _ in ms]))
    # AE-2 twin: the plaintext's true CRC (known, or what the plain decode yields when it yields anything)
    got = read(api, plain, verify_crc=0, ref_compat=0)
    true_crc = [zlib.crc32(r) if r is not None else (zlib.crc32(g[0]) if g[0] is not None else c) for (_, _, _, _, c, r), g in zip(ms, got)]
    plain2 = d / "plain_ae2.zip"
    plain2.write_bytes(aeszip.build_zip([aeszip.Entry(n, m, p, u, tc) for (n, m, p, u, _, _), tc in zip(ms, true_crc)]))
    enc = {}
    for vendor in (1, 2):
        for strength in (1, 2, 3):
            p = d / ("ae%d_s%d.zip" % (vendor, strength))
            p.write_bytes(aeszip.build_zip([aeszip.Entry(n, m, pl, u, c, strength, vendor, PW) for n, m, pl, u, c, _ in ms]))
            enc[vendor, strength] = p
    return ms, {1: plain, 2: plain2}, enc


@pytest.mark.parametrize("vendor", [1, 2])
@pytest.mark.parametrize("strength", [1, 2, 3])
def test_twin_archives(api, twins, vendor, strength):
    ms, plain, enc = twins
    for ref_compat in (0, 1):
        for verify_crc in (0, 1):
            a = read(api, enc[vendor, strength], PW, verify_crc, ref_compat)
            b = read(api, plain[vendor], None, verify_crc, ref_compat)
            for (name, *_), x, y in zip(ms, a, b):
                assert x == y, (name, ref_compat, verify_crc, hex(x[1]), hex(y[1]))


def test_twin_zipbomb_globals(api, twins):
    ms, plain, enc = twins
    ratio = C.c_uint64.in_dll(api.L, "otezip_max_expansion_ratio")
    slack = C.c_uint64.in_dll(api.L, "otezip_max_expansion_slack")
    old = ratio.value, slack.value, api.ignore_zipbomb.value
    try:
        for r, s, ig in ((3, 0, 0), (3, 0, 1), (50, 1000, 0)):
            ratio.value, slack.value, api.ignore_zipbomb.value = r, s, ig
            a = read(api, enc[2, 3], PW)
            b = read(api, plain[2])
            assert a == b, (r, s, ig)
            assert any(x[1] & 0xFF == 4 for x in a) or ig or r == 50
    finally:
        ratio.value, slack.value, api.ignore_zipbomb.value = old


def test_large_mixed_archive(api, tmp_path):
    rnd = random.Random(99)
    pool = synth.TextPool(8 << 20, 5)
    ents, raws = [], []
    sizes = [0, 1, 16 << 20] + [int(2 ** rnd.uniform(0, 17)) for _ in range(997)]
    for i, n in enumerate(sizes):
        raw = pool.take(n) if i % 3 else synth.random_bytes(n, i)
        meth = 8 if i % 4 else 0
        payload = synth.deflate_raw(raw, level=6) if meth == 8 else raw
        strength = (0, 1, 2, 3)[i % 4] if i != 2 else 3
        ents.append(aeszip.Entry("e%04d" % i, meth, payload, n, zlib.crc32(raw), strength, 1 + i % 2, PW))
        raws.append(raw)
    p = tmp_path / "mixed.zip"
    p.write_bytes(aeszip.build_zip(ents))
    got = read(api, p, PW, verify_crc=1)
    for e, r, (d, st) in zip(ents, raws, got):
        assert st == 0 and d == r, (e.name, hex(st))


def test_password_handling(api, tmp_path):
    raw = synth.jsonlog_text(200000, 7)
    comp = synth.deflate_raw(raw)
    mk = lambda pw, salt=None: aeszip.Entry("x", 8, comp, len(raw), zlib.crc32(raw), 3, 2, pw, salt)
    long_pw = bytes(range(33, 133))   # 100 bytes: hashed into the HMAC key first
    img = aeszip.build_zip([mk(PW), mk(b"other"), mk(long_pw), aeszip.Entry("plain", 0, raw, len(raw), zlib.crc32(raw))])
    p = tmp_path / "pw.zip"
    p.write_bytes(img)
    r = read(api, p)
    assert [x[1] for x in r[:3]] == [ST_NOPASSWD] * 3 and r[0][0] is None and r[3][0] == raw
    r = read(api, p, b"nope")
    assert [x[1] for x in r[:3]] == [ST_WRONGPASSWD] * 3 and r[3][0] == raw
    r = read(api, p, PW, per_entry={1: b"other", 2: long_pw})
    assert [x[0] for x in r] == [raw] * 4, [x[1] for x in r]
    # changing the default password between reads of the same open archive
    err = C.c_int(-1)
    za = api.L.zip_open(str(p).encode(), 0, C.byref(err))
    for pw, want in ((PW, raw), (b"other", None), (PW, raw), (None, None), (long_pw, None)):
        api.L.zip_set_default_password(za, pw)
        zf = api.L.zip_fopen_index(za, 0, 0)
        assert bool(zf) == (want is not None), pw
        if zf:
            assert C.string_at(zf.contents.data, zf.contents.size) == raw
            api.L.zip_fclose(zf)
    api.L.zip_set_default_password(za, b"other")
    zf = api.L.zip_fopen_index(za, 1, 0)
    assert zf and C.string_at(zf.contents.data, zf.contents.size) == raw
    api.L.zip_fclose(zf)
    assert not api.L.zip_fopen_index_encrypted(za, 1, 0, PW)
    api.L.zip_close(za)


def test_tampered_entries_are_never_handed_out(api, tmp_path):
    raw = synth.jsonlog_text(100000, 8)
    comp = synth.deflate_raw(raw)
    img = aeszip.build_zip([aeszip.Entry("x", 8, comp, len(raw), zlib.crc32(raw), 2, 1, PW, bytes(12))])
    lfh_data = 30 + 1 + 11
    sl = 12
    for where in (lfh_data + sl + 2 + 5000, lfh_data + sl + 2 + len(comp) + 3):   # a ciphertext bit, a code byte
        b = bytearray(img)
        b[where] ^= 0x10
        p = tmp_path / "t.zip"
        p.write_bytes(bytes(b))
        for vc in (0, 1):
            for rc in (0, 1):
                assert read(api, p, PW, vc, rc) == [(None, ST_AUTH)]
    # a payload too short to hold salt, verification value and code
    short = aeszip.build_zip([aeszip.Entry("s", 0, b"", 0, 0, 3, 2, PW)])
    cdo = struct.unpack_from("<I", short, len(short) - 6)[0]
    b = bytearray(short)
    struct.pack_into("<I", b, 18, 20)
    struct.pack_into("<I", b, cdo + 20, 20)
    p = tmp_path / "short.zip"
    p.write_bytes(bytes(b))
    assert read(api, p, PW) == [(None, ST_DATA_RANGE)]


def _write(api, path, files, pw=PW, default_pw=None, mode=ZIP_CREATE | ZIP_TRUNCATE):
    """files: (name, data, method, level, em or 0)"""
    err = C.c_int(-1)
    za = api.L.zip_open(str(path).encode(), mode, C.byref(err))
    assert za, err.value
    if default_pw is not None:
        api.L.zip_set_default_password(za, default_pw)
    keep = []
    for name, data, meth, lvl, em in files:
        buf = C.create_string_buffer(data, max(len(data), 1))
        keep.append(buf)
        src = api.L.zip_source_buffer(za, buf, len(data), 0)
        i = api.L.zip_file_add(za, name.encode(), src, 0)
        assert i >= 0
        assert api.L.zip_set_file_compression(za, i, meth, lvl) == 0
        if em:
            assert api.L.zip_file_set_encryption(za, i, em, pw if default_pw is None else None) == 0
    return api.L.zip_close(za)


def _files():
    ems = [ZIP_EM_AES_128, ZIP_EM_AES_192, ZIP_EM_AES_256]
    out = []
    k = 0
    for meth, lvl in ((0, 0), (8, 1), (8, 0), (93, 0)):
        for em in ems:
            for data in (synth.jsonlog_text(150000, k), synth.random_bytes(3000, k), b""):
                out.append(("f%02d" % k, data, meth, lvl, em))
                k += 1
    out.append(("plain", synth.jsonlog_text(5000, 99), 8, 0, 0))
    return out


@pytest.mark.parametrize("streaming", [0, 1])
def test_writer(api, tmp_path, streaming):
    zf_frames = C.c_int.in_dll(api.L, "otezip_zstd_frames")
    dd = C.c_int.in_dll(api.L, "otezip_write_data_descriptors")
    zf_frames.value, dd.value = 1, streaming
    try:
        files = _files()
        p = tmp_path / "w.zip"
        assert _write(api, p, files) == 0
        img = p.read_bytes()
        ents = aeszip.read_zip(img, PW)
        salts = set()
        for (name, data, meth, lvl, em), e in zip(files, ents):
            assert e["name"] == name
            if not em:
                assert e["aes"] is None and e["method"] == meth
                continue
            s = (em & 0xFF)
            assert e["method"] == 99 and e["flags"] & 1 and e["local_flags"] & 1 and e["local_method"] == 99
            assert e["aes"] == dict(vendor=2, strength=s, method=e["aes"]["method"]) and e["crc32"] == 0
            am = e["aes"]["method"]
            assert am in ((0,) if meth == 0 else (0, meth))
            if am == 93:
                from otezip_b200.zstdlib import Zstd
                assert Zstd().decompress(e["payload"], len(data)) == data
            else:
                assert aeszip.inflate(am, e["payload"]) == data
            assert bool(e["flags"] & 8) == bool(streaming)
            salts.add(e["raw"][:4 + 4 * s])
        assert len(salts) == sum(1 for f in files if f[4])
        with zipfile.ZipFile(p) as z:
            for f, info in zip(files, z.infolist()):
                assert bool(info.flag_bits & 1) == bool(f[4]) and (info.compress_type == 99) == bool(f[4])
        assert [d for d, _ in read(api, p, PW, verify_crc=1)] == [f[1] for f in files]
        # the same data written again gets new salts
        p2 = tmp_path / "w2.zip"
        assert _write(api, p2, files) == 0
        ents2 = aeszip.read_zip(p2.read_bytes())
        for e, e2 in zip(ents, ents2):
            if e["aes"]:
                assert e["raw"][:8] != e2["raw"][:8]
        # default password; appending plain entries keeps the encrypted ones byte for byte
        p3 = tmp_path / "w3.zip"
        assert _write(api, p3, files[:6], default_pw=b"dflt") == 0
        before = aeszip.read_zip(p3.read_bytes(), b"dflt")
        assert _write(api, p3, [("app", b"appended" * 100, 8, 0, 0)], mode=ZIP_CREATE) == 0
        after = aeszip.read_zip(p3.read_bytes(), b"dflt")
        assert [(x["raw"], x["aes"], x["flags"] & 1) for x in before] == [(x["raw"], x["aes"], x["flags"] & 1) for x in after[:6]]
        got = read(api, p3, b"dflt", verify_crc=1)
        assert [d for d, _ in got] == [f[1] for f in files[:6]] + [b"appended" * 100]
        # no password at all: zip_close fails instead of writing an entry it cannot encrypt
        assert _write(api, tmp_path / "np.zip", files[:1], pw=None) == -1
    finally:
        zf_frames.value, dd.value = 0, 0


def test_writer_more_than_65535_encrypted_entries(api, tmp_path):
    """One zip_close seals more entries than one call of the seam indexes passwords (65,534): ZIP64 directory, every entry
    under the default password, a few under their own."""
    n = 70000
    own = {5: b"five", 65540: b"late"}
    err = C.c_int(-1)
    p = tmp_path / "many.zip"
    za = api.L.zip_open(str(p).encode(), ZIP_CREATE | ZIP_TRUNCATE, C.byref(err))
    assert za
    api.L.zip_set_default_password(za, PW)
    keep = []
    for i in range(n):
        d = b"entry %d" % i
        buf = C.create_string_buffer(d, len(d))
        keep.append(buf)
        k = api.L.zip_file_add(za, b"m/%05d" % i, api.L.zip_source_buffer(za, buf, len(d), 0), 0)
        assert api.L.zip_file_set_encryption(za, k, ZIP_EM_AES_128 if i % 2 else ZIP_EM_AES_256, own.get(i)) == 0
    assert api.L.zip_close(za) == 0
    img = p.read_bytes()
    ents = aeszip.read_zip(img)
    assert len(ents) == n and all(e["method"] == 99 and e["aes"]["strength"] == (1 if i % 2 else 3) for i, e in enumerate(ents))
    for i in (0, 5, 65533, 65534, 65535, 65540, n - 1):
        e = ents[i]
        got = aeszip.open_payload(e["raw"], own.get(i, PW), e["aes"]["strength"])
        assert aeszip.inflate(e["aes"]["method"], got) == b"entry %d" % i
    r = read(api, p, PW, verify_crc=1, per_entry=own)
    assert [d for d, _ in r] == [b"entry %d" % i for i in range(n)]


CHILD = r'''
import ctypes as C, json, os, sys
sys.path.insert(0, %(root)r)
from otezip_b200.native import Lib
from tests import test_gpu_aes as T
from otezip_b200.zipapi import ZipApi
import tempfile, pathlib
api = ZipApi()
d = pathlib.Path(tempfile.mkdtemp())
ms = T._members()
from tests import aeszip
p = d / "e.zip"
p.write_bytes(aeszip.build_zip([aeszip.Entry(n, m, pl, u, c, 1 + i %% 3, 1 + i %% 2, T.PW) for i, (n, m, pl, u, c, _) in enumerate(ms)]))
T.read(api, p, T.PW)
C.c_int.in_dll(api.L, "otezip_zstd_frames").value = 1
assert T._write(api, d / "w.zip", T._files()) == 0
ok = [x for x, _ in T.read(api, d / "w.zip", T.PW)] == [f[1] for f in T._files()]
L = Lib.get().L
L.otz_debug_violations.argtypes = [C.c_void_p, C.c_int]
v = (C.c_uint64 * 32)()
n = L.otz_debug_violations(v, 32)
print(json.dumps({"slots": n, "violations": [int(x) for x in v[:max(n, 0)]], "roundtrip": ok}))
'''


def test_bounds_checked_build_counts_no_violation():
    dbg = os.path.join(ROOT, "otezip_b200", "libotezip_b200_dbg.so")
    if not os.path.exists(dbg):
        pytest.skip("debug library not built (make debug)")
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}], capture_output=True, text=True, timeout=1200, cwd=ROOT,
                       env=dict(os.environ, OTEZIP_B200_LIB=dbg))
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["slots"] > 0 and d["roundtrip"] and sum(d["violations"]) == 0, d
